// tower_f16.cu -- K3 tensor-core path for the residual tower (stem + 3 bottleneck blocks), fp16-split edition.
//
// Replaces the fp32 CUDA-core GEMMs of the tower (network.rs:65-125, network-utils lib.rs:386-461) with
// tcgen05.mma kind::f16, 3-pass hi/lo error compensation (x = fp16(x) + fp16(x - fp16(x)); lo.hi + hi.lo + hi.hi; see
// fc_f16.cu).  Per position the three 1x1 convolutions of a block are [81 x K] . [K x N] GEMMs with tiny K and N, so
// the design is about latency and data placement, not MMA throughput:
//   * the ACTIVATIONS are the A operand and live in TENSOR MEMORY (lane = pixel row, two fp16 channels per 32-bit
//     column, hi and lo parts of a 16-channel group side by side); threads write them with tcgen05.st straight
//     from registers (conv0, conv2).  conv1's A operand is the exception: the depthwise stencil runs on threads that own
//     a board row x a channel pair, so its outputs go to a no-swizzle K-major tile in SHARED memory (see T16_A_CHUNK);
//   * the WEIGHTS are the B operand in shared memory, K-major SWIZZLE_128B, hi and lo parts, scaled by a power of
//     two and pre-swizzled once on the device (k_tower16_pack), so one block's 36 KB image arrives by plain bulk
//     copies (cp.async.bulk) into a double buffer, one block ahead;
//   * the residual stream x stays in REGISTERS (a thread owns one pixel row x 64 channels) across all three blocks;
//     the depthwise 3x3 reads a small fp32 shared tile that epilogue 1 writes (the transposition pixel -> board row);
//   * a CTA PAIR (2x1 cluster) walks position TRIPLES: the 243 pixel rows of three positions fill 243 of the pair's
//     256 TMEM lanes.  The middle position straddles the two CTAs; the stencil band it needs from the peer is
//     mirrored through distributed shared memory;
//   * a CTA needs 256 TMEM columns, 111 KB of shared memory and <= 128 registers per thread, so TWO CTAs are
//     resident per SM: one CTA's MMA / barrier latencies hide behind the other's CUDA-core epilogues (the 3 x TF32
//     kernel this replaces needed all 512 columns and ran one 8-warp CTA per SM, every phase exposed).
// Warp w works on TMEM lane quadrant w%4 and channel set h = w/4 of the residual stream: channels [32h, 32h+32) and
// [64+32h, 64+32h+32) (x[0..31], x[32..63] of its threads) -- so that conv2's output columns [0,64) serve the FIRST pass of
// epilogue 3 of every warp and [64,128) the second: conv2 runs as two N = 64 halves with their own completion barriers
// (the second half's MMAs hide behind the first pass).  The elected thread of warp 0 issues the MMA chains.
//
// TMEM columns: X/D3 [0,128)  16-channel group kk of x: hi [16kk,16kk+8) lo [16kk+8,16kk+16); the conv2 accumulator
//                             D3 (fp32, 128 columns) aliases it: x's TMEM copy is dead once conv0 has read it
//               H    [128,160) 16-channel group g of the block's hidden activations, same hi/lo packing
//               ACC  [160,192) the conv0 / conv1 accumulator (fp32, 32 columns)
//               ONE  [192,200) constant A group of the bias MMA (k = 0, 1: 64.0; k = 2..15: 0); [200,256) unused (allocations are powers of two)
#include <cstdio>
#include <cstdlib>

#include "omk_internal.h"
#include "tc_ptx.cuh"

namespace omk {

using namespace tc;

constexpr int T16_THREADS = 256;
constexpr uint32_t T16_TMEM_COLS = 256;
constexpr uint32_t TC_X = 0, TC_D3 = 0, TC_H = 128, TC_ACC = 160, TC_ONE = 192;  // TC_ONE: 8 columns, the bias MMA's constant A group
// per-block weight image (bytes).  W0^T [32 n][128 k]: hi and lo, each two k-atoms of [32 rows x 128 B];
// PW^T [32 n][32 k] and W2^T [128 n][32 k]: hi in bytes [0,64) and lo in bytes [64,128) of each 128-byte row
// (the three bias tiles sit between W0 and PW so that, once conv0 has read W0 and its bias tile, bytes [0, 16896) of the
// image are dead for the rest of the block: the row stencil's A tile lives there)
constexpr int W16_W0HI = 0, W16_W0LO = 8192, W16_PW = 19456, W16_W2 = 23552;
// conv2's bias b2 goes THROUGH THE MMA: one extra k-step whose A operand is a constant group of TMEM columns (k = 0, 1 hold
// T16_BIAS_ONE, the rest zero) and whose B operand is this tile: [128 n][8 k] fp16, K-major WITHOUT swizzle (core matrices
// of 8 rows x 16 bytes), k = 0 / 1 = hi / lo halves of b2[n] * 2^s / T16_BIAS_ONE.  The second k-chunk of the K = 16
// instruction points (leading-byte-offset) at a block of zeros shared by both weight buffers.  Epilogue 3 then is
// x = lrelu(d * 2^-s + x): per channel pair one FFMA2 instead of FFMA2 + FADD2 and no constant-bank load of the bias; epilogues
// 1 and 2 are lrelu(d * 2^-s) = max(d * 2^-s, d * 0.2 * 2^-s) in packed fp32x2 multiplies, no bias operand at all.
constexpr int W16_B0T = 16384, W16_B1T = 16896;  // conv0 / conv1: [32 n][8 k] each (the same construction for b0 and b1)
constexpr int W16_B2T = 17408;                   // conv2: [128 n][8 k]
constexpr int W16_BYTES = 36864 + 2048 + 1024;
static_assert(W16_PW == W16_B2T + 2048 && W16_PW % 1024 == 0 && W16_W2 == W16_PW + 4096 && W16_BYTES == W16_W2 + 16384, "weight image layout");
// ROW STENCIL (default; -DOMK_T16_PIXEL_STENCIL builds the previous form for A/B).  The depthwise 3x3 is computed by threads
// that own a BOARD ROW x a CHANNEL PAIR (a half-warp = one board row x 32 channels) instead of a pixel x 16 channels: a thread
// slides over the nine columns of its row, loads each input (three rows x nine columns, one LDS.64 each: 27 loads for 9
// outputs x 2 channels instead of 9 neighbour rows x 16 channels = 36 LDS.128 for one pixel) and accumulates into the three
// outputs it touches with packed fp32x2 FMAs whose weight operands are nine register pairs.  Shared-memory wavefronts of the
// phase: 8 warps x 54 instead of 8 x 144.  The outputs leave as fp16 hi / lo straight into conv1's A OPERAND IN SHARED MEMORY
// (the transposition back to "lane = pixel" that tensor memory would need is free there): K-major without swizzle, core
// matrices of 8 pixel rows x 16 bytes, 8-row groups contiguous (SBO = 128), so a pixel row R of k-chunk c sits at
// c * T16_A_CHUNK + 16 R -- affine in R, every store offset is an immediate -- and the chunk stride of 2048 + 32 bytes spreads
// a half-warp's four k-chunks (and the other half-warp's row, nine pixels on) over all 32 banks: one wavefront per STS.32.
// Chunks 0..3: hi of channels 8c..8c+7, chunks 4..7: lo.
constexpr int T16_A_CHUNK = 2080, T16_A_BYTES = 7 * T16_A_CHUNK + 2048;
static_assert(T16_A_BYTES <= W16_B1T, "the A tile overlays W0 hi / lo and conv0's bias tile only");
#ifdef OMK_T16_PIXEL_STENCIL
constexpr bool T16_ROWS = false;
#else
constexpr bool T16_ROWS = true;
#endif
constexpr float T16_BIAS_ONE = 64.0f;  // |b2| up to 65504 * 64 / 2^s stays finite in the fp16 tile
// The small fp32 parameters travel as a KERNEL ARGUMENT (7.9 KB of the constant bank): every use is warp-uniform, so
// biases, stem and depthwise weights become constant-bank operands of the FMAs instead of shared-memory loads.
struct alignas(16) Tower16Block {
    float b0[32], dw[9][32], b1[32], b2[128];
    float inv[4];  // 2^-s of w0, pw, w2 (undo the power-of-two weight scaling; exact)
};
struct alignas(16) Tower16Params {
    float wstem[3][128], bstem[128];
    Tower16Block blk[3];
};
// the same image as plain floats (k_tower16_pack writes it on the device; the host keeps a copy to pass by value)
constexpr int P16_WSTEM = 0, P16_BSTEM = 384, P16_BLK0 = 512, P16_BLK = 484;
constexpr int P16_B0 = 0, P16_DW = 32, P16_B1 = 320, P16_B2 = 352, P16_INV = 480;
constexpr int P16_FLOATS = P16_BLK0 + 3 * P16_BLK;  // 1964
static_assert(sizeof(Tower16Params) == P16_FLOATS * 4 && sizeof(Tower16Block) == P16_BLK * 4, "parameter image layout");
constexpr int T16_HSTRIDE = 36;                     // fp32 depthwise tile row stride (floats): conflict-free float4 rows
// shared memory map (bytes from the 1024-aligned base)
constexpr int S16_W = 0;                                      // 2 x 38 KB weight images
constexpr int S16_ZERO = 2 * W16_BYTES;                       // 2 KB of zeros (second k-chunk of the bias MMAs)
constexpr int S16_H = S16_ZERO + 2048;                        // [162 rows (two positions)][36] fp32
constexpr int S16_IMG = S16_H + 162 * T16_HSTRIDE * 4;        // three 243-float input images (boards path: block 0's conv0 table)
constexpr int S16_TAB = S16_IMG + 736 * 4;                    // fp32 stem table, 8 input combinations x 132 words
constexpr int T16_TABSTRIDE = 132;                            // words per combination: 128 + 4, so the 8 rows start 4 banks apart
// (the PACKED hi/lo stem table is needed only once, for the conv0 table at kernel start: it borrows the depthwise tile)
constexpr int S16_BAR = S16_TAB + 8 * T16_TABSTRIDE * 4;
constexpr int T16_SMEM_BYTES = S16_BAR + 64 + 1024;           // 111 KB: two CTAs per SM (2 x (smem + 1 KB) <= 228 KB)
// ... and stays clear of the rows the PEER may already mirror into this tile while the table is still being read: the peer's
// band lands in rows >= 37 (rank 0 writes its pixels 37..80 of slot 0's position, rank 1 rows 81 + p)
static_assert(8 * T16_TABSTRIDE * 4 <= 37 * T16_HSTRIDE * 4, "the packed stem table fits below the first mirrored band row of the tile it borrows");
static_assert(2 * (T16_SMEM_BYTES + 1024) <= 233472, "two CTAs per SM");
constexpr uint32_t T16_BAND_BYTES = 10 * 32 * 4;              // mirrored stencil band: 10 pixel rows x 32 channels fp32
constexpr uint32_t T16_IDESC_N32 = idesc_f16(128, 32), T16_IDESC_N64 = idesc_f16(128, 64), T16_IDESC_N128 = idesc_f16(128, 128);
#ifdef OMK_T16_NO_SPLIT2
constexpr bool T16_SPLIT2 = false;   // conv2 as one N = 128 chain (A/B)
#else
constexpr bool T16_SPLIT2 = true;
#endif
static_assert(W16_BYTES >= 8 * 4608 && W16_BYTES % 64 == 0, "the idle weight buffer doubles as eight per-warp staging tiles (4 KB used, 512-byte aligned)");
static_assert(S16_BAR % 8 == 0, "mbarriers are 8-byte aligned");

__device__ long long g_t16_dbg[64];  // phase timestamps of CTA 0's second iteration (omk_debug_tower_timing)
// Phase timestamps exist only in the STAMPS instantiation (env OMK_TOWER_STAMPS=1, tests/tools/check_f16.py): even
// predicated off, the 25 clock reads + stores cost 4 % of the kernel.
#define T16_STAMP(i) do { if constexpr (STAMPS) { if (dbg_on && t == 0) g_t16_dbg[(i)] = clock64(); } } while (0)
// Wait for one of the CTA's mbarriers.  ONE warp polls it, the others block on the CTA barrier (no issue slots): with all
// eight warps polling, try_wait + branch pairs were 10 % of the kernel's issued instructions.
#define T16_WAIT(bar, parity) do { if (warp == 7) mbar_wait((bar), (parity)); __syncthreads(); } while (0)
#ifdef OMK_T16_ALLPOLL
#define T16_WAIT_MMA(bar, parity) mbar_wait((bar), (parity))
#else
#define T16_WAIT_MMA(bar, parity) T16_WAIT(bar, parity)
#endif
__device__ __forceinline__ float t16_lrelu(float v) { return fmaxf(v, 0.2f * v); }  // alpha < 1: max(v, alpha v)

// split 16 fp32 values (one 16-channel group) into 8 packed hi words + 8 packed lo words and store them as A-operand columns
__device__ __forceinline__ void t16_store_group(uint32_t taddr, const float *v) {
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) split2_f16(v[2 * i], v[2 * i + 1], w[i], w[8 + i]);
    tmem_st16(taddr, w);
}

// TMA write-out of one warp's 32 pixel rows x 64 channels as fp16 hi / lo (the A operand of fc0).  The arrays are viewed as
// [triple][243 pixel rows][128 channels]: the pair's rows are one contiguous block, a warp's piece of it is a box of 32
// rows x 32 channels (64 bytes) per pass, hi and lo, and the pair's 13 padding rows (>= 243) are clipped by the tensor map.
// The warp stages the box in its 4 KB tile of the idle weight buffer in the SWIZZLE_64B pattern (16-byte chunk index ^=
// (row >> 1) & 3: conflict-free stores) and one lane issues cp.async.bulk.tensor stores: no per-thread global stores, no
// LSU queue to drain before the next iteration's first shared-memory load (the per-thread STG.128 form -- 16 per thread,
// eight 64-byte segments per instruction -- cost 11 % of the kernel in L1 tag cycles).
// One pass = 32 channels (x32) of the warp's 32 rows; the caller makes sure the previous pass's stores have read the tile.
__device__ __forceinline__ void t16_store_pass(uint32_t tile, int lane, const float *x32, const CUtensorMap *map_hi,
                                               const CUtensorMap *map_lo, int ch, int r0, int tr) {
    const uint32_t rowoff = (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        uint4 h, l;
        const float *v = x32 + k * 8;
        split2_f16(v[0], v[1], h.x, l.x);
        split2_f16(v[2], v[3], h.y, l.y);
        split2_f16(v[4], v[5], h.z, l.z);
        split2_f16(v[6], v[7], h.w, l.w);
        const uint32_t a = tile + rowoff + (((uint32_t)k ^ sw) << 4);
        sts128(a, h);
        sts128(a + 2048u, l);
    }
    fence_proxy_async_smem();  // generic-proxy writes -> visible to the TMA engine
    __syncwarp();
    if (lane == 0) {
        tma_store_3d(map_hi, tile, ch, r0, tr);
        tma_store_3d(map_lo, tile + 2048u, ch, r0, tr);
        bulk_commit();
    }
}

// ---- per-phase CUDA-core work, templated on the channel half so that every parameter offset is a compile-time
//      constant-bank address (the half is warp-uniform but the compiler cannot prove it).  Measured: indexing by a run-time
//      half instead shrinks the kernel from 4.9k to 3.9k SASS instructions but runs 9 % slower. ----
// stem 1x1 conv 3 -> 128 (network.rs:65-79): this thread's pixel, its 64 channels
template <int HALF>
__device__ __forceinline__ void t16_stem(const Tower16Params &P, float v0, float v1, float v2, float *x) {
#pragma unroll
    for (int c = 0; c < 64; c += 2) {
        const int ch = HALF * 32 + c + (c >= 32 ? 32 : 0);  // x[c] is channel t16_chan(HALF, c)
        float2 s = __ffma2_rn(make_float2(v0, v0), make_float2(P.wstem[0][ch], P.wstem[0][ch + 1]),
                              make_float2(P.bstem[ch], P.bstem[ch + 1]));
        s = __ffma2_rn(make_float2(v1, v1), make_float2(P.wstem[1][ch], P.wstem[1][ch + 1]), s);
        s = __ffma2_rn(make_float2(v2, v2), make_float2(P.wstem[2][ch], P.wstem[2][ch + 1]), s);
        x[c + 0] = t16_lrelu(s.x);
        x[c + 1] = t16_lrelu(s.y);
    }
}
// epilogue 1 / 2 arithmetic: lrelu(acc * 2^-s + bias).  Scalar on purpose: the packed fp32x2 forms measured 7 % slower here
// (operands not in aligned register pairs), while in the stem / stencil / residual / split code, where pairs are natural,
// scalar forms measured 1-5 % slower.
// History of the accumulator chains: with the MMA loop rolled and its operands in vector registers, ptxas wrapped every
// tcgen05.mma in ~30 instructions of elect / R2UR waterfall code (~175 clk per dependent MMA), and three parallel chains per
// convolution (one per product, three partial accumulators added here) beat a single chain by 14 %.  With warp-uniform
// operands and unrolled chains the MMAs issue back to back (tower 0.749 -> 0.658 ms) and ONE chain per convolution is
// faster again (0.648 ms): two TMEM loads and two adds per element less in each of these epilogues.
// (the bias is in the accumulator: it went through the MMA as one more k-step)
__device__ __forceinline__ void t16_lrelu_scaled16(float inv, const float *d, float *o) {
    const float2 i2 = make_float2(inv, inv), j2 = make_float2(0.2f * inv, 0.2f * inv);  // 0.2 * 2^-s is exact up to fp32(0.2)
#pragma unroll
    for (int c = 0; c < 16; c += 2) {
        const float2 v = make_float2(d[c], d[c + 1]);
        const float2 a = __fmul2_rn(v, i2), b = __fmul2_rn(v, j2);
        o[c] = fmaxf(a.x, b.x);
        o[c + 1] = fmaxf(a.y, b.y);
    }
}
// depthwise 3x3, SAME zero padding, no bias (lib.rs:204-216): 16 channels of pixel (y, x0) from the fp32 tile.
// (Measured and rejected, twice: branch-free variants whose off-board taps read zeros.  The second one used a zero-padded
// tile -- board rows of [128 zero bytes | 9 x 144-byte entries], every tap the centre plus a constant, no bank conflicts
// (a first padded layout with 144-byte zero entries had 2-way conflicts at every board-row boundary: +10 %) -- and, with
// ~100 fewer instructions per warp and block, still ran 5 % slower than the per-tap bounds tests: the phase is bound by the
// 144 shared-memory wavefronts per warp of the neighbour rows, not by its instruction count.  Taking the centre tap from
// the thread's own epilogue-1 registers instead of the tile (four loads less) was 6 % slower: sixteen more live registers
// across the band barrier.  Loading the fp32 residual rows of the stem table behind block 0's conv2 instead of in the stem
// phase: 20 % slower -- this kernel lives at 128 registers and every change of live ranges shows.)
template <int HALF>
__device__ __forceinline__ void t16_stencil(const Tower16Block &B, const float *Hpos /* tile rows of this position */, int y, int xx0,
                                            float *a) {
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int yy = y + ky - 1;
        if (yy < 0 || yy >= kSide) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int xx = xx0 + kx - 1;
            if (xx < 0 || xx >= kSide) continue;
            const float *hp = Hpos + (yy * kSide + xx) * T16_HSTRIDE + HALF * 16;
#pragma unroll
            for (int c = 0; c < 16; c += 4) {
                const float4 h = *reinterpret_cast<const float4 *>(hp + c);
                const float4 w = *reinterpret_cast<const float4 *>(&B.dw[ky * 3 + kx][HALF * 16 + c]);  // one LDCU.128
                // packed fp32x2 FMA (sm_100): same results as two FFMAs, half the issue slots
                const float2 lo2 = __ffma2_rn(make_float2(h.x, h.y), make_float2(w.x, w.y), make_float2(a[c + 0], a[c + 1]));
                const float2 hi2 = __ffma2_rn(make_float2(h.z, h.w), make_float2(w.z, w.w), make_float2(a[c + 2], a[c + 3]));
                a[c + 0] = lo2.x; a[c + 1] = lo2.y; a[c + 2] = hi2.x; a[c + 3] = hi2.y;
            }
        }
    }
}
// epilogue 3 arithmetic on 32 channels [c0, c0+32) of this thread's 64: x = lrelu(d * 2^-s + b2 + x)
template <int HALF>
__device__ __forceinline__ void t16_residual32(const Tower16Block &B, int c0, const float *d, float *x) {
    const float inv = B.inv[2];  // (the accumulator already holds (conv2 + b2) * 2^s: the bias went through the MMA)
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        const int c = c0 + i;
        const float2 tt = __ffma2_rn(make_float2(d[i], d[i + 1]), make_float2(inv, inv), make_float2(x[c], x[c + 1]));
        const float2 u = __fmul2_rn(tt, make_float2(0.2f, 0.2f));
        x[c + 0] = fmaxf(tt.x, u.x);
        x[c + 1] = fmaxf(tt.y, u.y);
    }
}
// The three input floats of one pixel as bits.  The reference's 243-float slot (encoder.rs:22-43) read as [81][3] puts
// floats 3 pc .. 3 pc + 2 at pixel pc: for pc < 54 they are (cell, plane) entries f -> (f >> 1, f & 1) of the interleaved
// stone planes -- two neighbouring cells A, B = A + 1 -- and for pc >= 54 (f >= 162) all three lie in the turn plane.
// Which words of the request row a thread needs never changes, so it loads just those (5 words instead of the 32-byte
// row) and the per-iteration work is a handful of shifts and selects (same values as image_value()).
struct T16Req { uint32_t bA, wA, bB, wB, meta; };
struct T16ReqSpec { int wordA, wordB; uint32_t sA, sB, odd, turn; };  // thread-invariant
__device__ __forceinline__ T16ReqSpec t16_req_spec(int pc) {
    T16ReqSpec q;
    q.turn = pc >= 54;
    const int f0 = q.turn ? 0 : 3 * pc, cA = f0 >> 1, cB = cA + 1;
    q.wordA = cA >> 5; q.sA = cA & 31; q.wordB = cB >> 5; q.sB = cB & 31; q.odd = f0 & 1;
    return q;
}
__device__ __forceinline__ T16Req t16_req_load(const NNIn *row, const T16ReqSpec &q) {
    const uint32_t *rp = reinterpret_cast<const uint32_t *>(row);
    T16Req r;
    r.bA = rp[q.wordA]; r.wA = rp[3 + q.wordA]; r.bB = rp[q.wordB]; r.wB = rp[3 + q.wordB]; r.meta = rp[6];
    return r;
}
__device__ __forceinline__ uint32_t t16_req_combo(const T16Req &r, const T16ReqSpec &q) {
    const uint32_t bA = (r.bA >> q.sA) & 1u, wA = (r.wA >> q.sA) & 1u, bB = (r.bB >> q.sB) & 1u, wB = (r.wB >> q.sB) & 1u;
    const uint32_t persp = (r.meta ^ (r.meta >> 1)) & 1u;  // EnvTurnMode::Opponent flips the perspective
    // plane k holds black where k == persp.  even f0: (A, 0) (A, 1) (B, 0); odd f0: (A, 1) (B, 0) (B, 1)
    const bool e = (q.odd ^ persp) != 0;              // "plane (f0 & 1) is the white one"
    const uint32_t bY = q.odd ? bB : bA, wY = q.odd ? wB : wA;
    const uint32_t ch0 = e ? wA : bA, ch1 = e ? bY : wY, ch2 = e ? wB : bB;
    const uint32_t stones = ch0 | (ch1 << 1) | (ch2 << 2);
    return q.turn ? ((r.meta & 1u) ^ 1u) * 7u : stones;  // turn plane: 1.0 when black is to move
}
__device__ __forceinline__ float2 t16_lds64(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));  // volatile: stays behind the barrier it follows
    return v;
}
__device__ __forceinline__ void t16_sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// Row stencil: depthwise 3x3 (SAME zero padding, no bias; lib.rs:204-216) of one board row x one channel pair.  `up`, `mid`,
// `dn` address the three input rows in the fp32 tile (a row off the board points at the shared block of zeros: the taps
// then add 0 * w, exactly); w[ky * 3 + kx] are this thread's nine weight pairs.  Output column xo of the row is pixel row
// r0 + xo of the CTA's 128 (stored when it is one of them: the pair's middle position straddles the CTAs) and goes to
// conv1's A tile as packed fp16 hi (chunk c) / lo (chunk 4 + c) words.
__device__ __forceinline__ void t16_row_stencil(uint32_t up, uint32_t mid, uint32_t dn, const float2 *w, uint32_t a_addr, int r0) {
    // (all loads and FMAs first, the splits and stores after: a store between the columns would pin every later load behind it)
    float2 o[kSide];
    constexpr uint32_t PX = T16_HSTRIDE * 4;
#pragma unroll
    for (int xi = 0; xi < kSide; ++xi) {
        const float2 i0 = t16_lds64(up + xi * PX), i1 = t16_lds64(mid + xi * PX), i2 = t16_lds64(dn + xi * PX);
        // input column xi is the kx = 2 tap of output xi - 1, the kx = 1 tap of output xi, the kx = 0 tap of output xi + 1
        if (xi > 0) {
            o[xi - 1] = __ffma2_rn(i0, w[2], o[xi - 1]); o[xi - 1] = __ffma2_rn(i1, w[5], o[xi - 1]); o[xi - 1] = __ffma2_rn(i2, w[8], o[xi - 1]);
        }
        // (output xi's first tap is its kx = 0 one, from column xi - 1, except in column 0)
        o[xi] = xi > 0 ? __ffma2_rn(i0, w[1], o[xi]) : __fmul2_rn(i0, w[1]);
        o[xi] = __ffma2_rn(i1, w[4], o[xi]); o[xi] = __ffma2_rn(i2, w[7], o[xi]);
        if (xi + 1 < kSide) {
            o[xi + 1] = __fmul2_rn(i0, w[0]);
            o[xi + 1] = __ffma2_rn(i1, w[3], o[xi + 1]); o[xi + 1] = __ffma2_rn(i2, w[6], o[xi + 1]);
        }
    }
#pragma unroll
    for (int xo = 0; xo < kSide; ++xo) {
        uint32_t hi, lo;
        split2_f16(o[xo].x, o[xo].y, hi, lo);
        const int R = r0 + xo;
        if (R >= 0 && R < 128) {
            t16_sts32(a_addr + (uint32_t)(xo * 16), hi);
            t16_sts32(a_addr + (uint32_t)(xo * 16 + 4 * T16_A_CHUNK), lo);
        }
    }
}
// first channel of x[c .. c + 15] (c a multiple of 16) of a thread with channel set h
__device__ __forceinline__ int t16_chan(int h, int c) { return 32 * h + c + (c >= 32 ? 32 : 0); }
// conv0's accumulator chain over the 8 k-groups of X plus the bias step (one elected thread; all operands warp-uniform).
// (Measured and rejected: issuing k-groups 0..3 of the NEXT block's conv0 from the middle of epilogue 3, once every warp's
// first pass is in tensor memory -- warp 0 then waits for the slowest warp before its own second pass: +-0.)
__device__ __forceinline__ void t16_issue_conv0(uint32_t tmem_base, uint32_t wb, uint32_t zero) {
    constexpr int K0 = 0, K1 = 8;
    const uint64_t bhi = desc_sw128(wb + W16_W0HI), blo = desc_sw128(wb + W16_W0LO);
    const uint32_t dcol = tmem_base + TC_ACC;
#pragma unroll
    for (int kk = K0; kk < K1; ++kk) {
        const uint64_t off = (uint64_t)(((kk >> 2) * 4096 + (kk & 3) * 32) >> 4);
        const uint32_t ahi = tmem_base + TC_X + 16u * kk;
        umma_f16_ts(dcol, ahi + 8u, bhi + off, T16_IDESC_N32, kk != 0);
        umma_f16_ts(dcol, ahi, blo + off, T16_IDESC_N32, 1u);
        umma_f16_ts(dcol, ahi, bhi + off, T16_IDESC_N32, 1u);
    }
    if (K1 == 8)
        umma_f16_ts(dcol, tmem_base + TC_ONE, desc_nosw(wb + W16_B0T, zero - (wb + W16_B0T), 128u), T16_IDESC_N32, 1u);  // + b0
}
#define T16_HALF(call_0, call_1) do { if (half == 0) { call_0; } else { call_1; } } while (0)

// BOARDS: the hot path (packed request rows).  Block 0's conv0 + epilogue 1 are then a TABLE as well: the stem output of a
// pixel is one of 8 rows, so conv0(stem row) + b0, lrelu is one of 8 rows of 32 channels.  Each CTA computes those 8 rows
// once, at kernel start, THROUGH THE SAME MMA CHAIN AND EPILOGUE ARITHMETIC as the general path (TMEM lanes 0..7 = the 8
// packed stem rows; a row of D depends only on its own row of A), so the boards path stays bit-identical to the float-image
// path (tested).  Per iteration that removes the stem's 128-channel operand store, block 0's conv0 MMA round trip and the
// arithmetic of its epilogue 1.
template <bool STAMPS, bool BOARDS>
__global__ void __launch_bounds__(T16_THREADS, 2)
    k_tower16(const uint8_t *__restrict__ wimg, const __grid_constant__ Tower16Params P, const NNIn *__restrict__ nn_in,
              const float *__restrict__ images, const uint32_t *n_req, int max_rows, const __grid_constant__ CUtensorMap map_hi,
              const __grid_constant__ CUtensorMap map_lo, const float *__restrict__ pimg) {
    extern __shared__ uint8_t t16_smem_raw[];
    // (the broadcasts below tell ptxas that these values are warp-uniform: the MMA issue code then runs on uniform registers)
    const int rows = __shfl_sync(0xffffffffu, (int)min(*n_req, (uint32_t)max_rows), 0);
    const int n_triples = (rows + 2) / 3, n_pairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
    if (pair >= n_triples) return;  // uniform for both CTAs of the pair, before any cluster barrier
    const uint32_t rank = cluster_rank();
    const int t = threadIdx.x, warp = __shfl_sync(0xffffffffu, t >> 5, 0), lane = t & 31;
    const int q = warp & 3, half = warp >> 2;
    // Row R of the pair = 128*rank + TMEM lane; position j = R/81, pixel p = R%81.
    const int R = (int)rank * 128 + q * 32 + lane;
    const int j = R / kCells, p = R - j * kCells;
    const int slot = j - (int)rank;  // H tile slot: CTA r keeps positions r and r+1 (162 rows)
    const bool in_tile = R < 3 * kCells;
    // The pair's middle position straddles the two CTAs.  The H rows of it that the PEER's stencil reaches (pixels 37..46
    // held by CTA 0, 47..56 held by CTA 1) are mirrored into the peer's tile with st.async, which signals the peer's
    // "band" mbarrier by transaction bytes: no cluster-wide barrier and no fence in the loop.
    const bool band = j == 1 && (rank == 0 ? p >= 37 : p <= 56);
    // Row stencil: half-warp (warp, lane >> 4) owns board-row unit 2 * warp + (lane >> 4) of this CTA's 128 pixel rows --
    // rank 0: position 0 rows 0..8, position 1 rows 0..5 (row 5: its first two pixels); rank 1: position 1 rows 5..8 (row 5:
    // the other seven), position 2 rows 0..8 -- and the lane's channel pair.  Row 5 of the middle position is computed by
    // both CTAs, each storing its own pixels; the inputs those need are its own rows and the mirrored band, as before.
    const int unit = warp * 2 + (lane >> 4), cp = lane & 15;
    const bool has_unit = unit < (rank == 0 ? 15 : 13);
    const int uj = rank == 0 ? (unit >= 9 ? 1 : 0) : (unit < 4 ? 1 : 2);
    const int urow = rank == 0 ? (unit >= 9 ? unit - 9 : unit) : (unit < 4 ? unit + 5 : unit - 4);

    uint8_t *sm = t16_smem_raw + ((1024u - (smem_u32(t16_smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(sm);
    float *H0 = reinterpret_cast<float *>(sm + S16_H);
    float *T32 = reinterpret_cast<float *>(sm + S16_TAB);
    float *IMG = reinterpret_cast<float *>(sm + S16_IMG);
    float *T0 = IMG;  // boards path: block 0's conv0 table, 8 rows x T16_HSTRIDE floats (the image buffer is unused there)
    uint32_t *TW = reinterpret_cast<uint32_t *>(sm + S16_H);  // packed stem table: used once, before the tile is
    const uint32_t bar_w0 = sbase + S16_BAR, bar_mma = sbase + S16_BAR + 16, bar_band = sbase + S16_BAR + 24,
                   bar_free = sbase + S16_BAR + 32, tmem_slot = sbase + S16_BAR + 40, bar_mma2 = sbase + S16_BAR + 48;
    const uint32_t peer_h0 = mapa(sbase + S16_H, rank ^ 1u);
    const uint32_t peer_band = mapa(bar_band, rank ^ 1u), peer_free = mapa(bar_free, rank ^ 1u);

    if (t == 0) {
        mbar_init(bar_w0, 1);
        mbar_init(bar_w0 + 8, 1);
        mbar_init(bar_mma, 8);   // one tcgen05.commit per warp
        mbar_init(bar_band, 1);  // one arrive.expect_tx per block + the peer's 1280 mirrored bytes
        mbar_init(bar_free, 1);  // the peer's "I have read your band" arrival
        mbar_init(bar_mma2, 1);  // conv2's second half (one commit by the issuing thread)
        mbar_fence_init();
    }
    // Stem tables.  A board's input pixel is one of 8 bit triples (encoder.rs:22-43 writes only 0.0 / 1.0), so the stem
    // 3 -> 128 convolution + lrelu of a pixel is one of 8 rows: each CTA computes them once, with the arithmetic of
    // t16_stem (bit-identical to the general float-image path), as fp32 and as packed fp16 hi / lo A-operand words.
    for (int e = t; e < 2048 / 16; e += T16_THREADS) reinterpret_cast<uint4 *>(sm + S16_ZERO)[e] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's shared-memory reads (before the barriers below)
    for (int e = BOARDS ? t : 8 * 64; e < 8 * 64; e += T16_THREADS) {
        const int combo = e >> 6, ch = (e & 63) * 2;
        const float v0 = (float)(combo & 1), v1 = (float)((combo >> 1) & 1), v2 = (float)(combo >> 2);
        float2 sv = __ffma2_rn(make_float2(v0, v0), make_float2(P.wstem[0][ch], P.wstem[0][ch + 1]),
                               make_float2(P.bstem[ch], P.bstem[ch + 1]));
        sv = __ffma2_rn(make_float2(v1, v1), make_float2(P.wstem[1][ch], P.wstem[1][ch + 1]), sv);
        sv = __ffma2_rn(make_float2(v2, v2), make_float2(P.wstem[2][ch], P.wstem[2][ch + 1]), sv);
        const float a0 = t16_lrelu(sv.x), a1 = t16_lrelu(sv.y);
        T32[combo * T16_TABSTRIDE + ch] = a0;
        T32[combo * T16_TABSTRIDE + ch + 1] = a1;
        uint32_t hi, lo;
        split2_f16(a0, a1, hi, lo);
        TW[combo * T16_TABSTRIDE + (ch >> 4) * 16 + ((ch & 15) >> 1)] = hi;  // group layout of t16_store_group: hi[8] then lo[8]
        TW[combo * T16_TABSTRIDE + (ch >> 4) * 16 + 8 + ((ch & 15) >> 1)] = lo;
    }
    if (warp == 1) tmem_alloc<1>(tmem_slot, T16_TMEM_COLS);
    fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's barriers exist before anything crosses the pair
    fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);  // this warp's lane quadrant

    {   // the bias MMA's constant A group: k = 0, 1 = T16_BIAS_ONE, k = 2 .. 15 = 0 (every lane; written once)
        uint32_t one8[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        const __half2 o2 = __floats2half2_rn(T16_BIAS_ONE, T16_BIAS_ONE);
        one8[0] = *reinterpret_cast<const uint32_t *>(&o2);
        tmem_st8(tlane + TC_ONE, one8);
        tmem_wait_st();
    }
    uint32_t g = 0;          // running block counter: weight buffer = g & 1, its phase parity = (g >> 1) & 1
    uint32_t mma_uses = 0;   // completed uses of bar_mma
    auto issue_weights = [&](uint32_t gg) {  // one thread
        const uint32_t buf = gg & 1u, bar = bar_w0 + 8 * buf;
        fence_proxy_async_smem();  // the buffer may have served as a staging tile (generic proxy)
        mbar_expect_tx(bar, (uint32_t)W16_BYTES);
        const uint8_t *src = wimg + (size_t)(gg % 3u) * W16_BYTES;
        for (int c = 0; c < W16_BYTES; c += W16_BYTES / 4) bulk_load(sbase + S16_W + buf * W16_BYTES + c, src + c, W16_BYTES / 4, bar);
    };
    if (t == 0) issue_weights(0);

    if constexpr (BOARDS) {
        // ---- block 0's conv0 table: the 8 packed stem rows through conv0's MMA chain and epilogue 1, once per CTA ----
        if (warp == 0) {  // TMEM lanes 0..7 <- packed rows (lanes >= 8 repeat row 7: their accumulator rows are never read)
            const uint4 *tw = reinterpret_cast<const uint4 *>(TW + min(lane, 7) * T16_TABSTRIDE);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint32_t w[16];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint4 v = tw[c * 4 + k];
                    w[4 * k + 0] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
                }
                tmem_st16(tlane + TC_X + (uint32_t)(c * 16), w);
            }
            tmem_wait_st();
        }
        fence_before();
        __syncthreads();
        if (warp == 0) {
            if (elect_one()) {
                fence_after();
                mbar_wait(bar_w0, 0u);
                t16_issue_conv0(tmem_base, sbase + S16_W, sbase + S16_ZERO);  // the same chain as conv0 in the loop below
                umma_commit(bar_mma);
            }
        } else if (lane == 0) {
            fence_after();
            umma_commit(bar_mma);
        }
        T16_WAIT(bar_mma, mma_uses & 1u);
        ++mma_uses;
        fence_after();
        if (warp == 0) {
            float d[32], o[32];
            tmem_ld16(tlane + TC_ACC, d);
            tmem_ld16(tlane + TC_ACC + 16, d + 16);
            tmem_wait_ld();
            t16_lrelu_scaled16(P.blk[0].inv[0], d, o);
            t16_lrelu_scaled16(P.blk[0].inv[0], d + 16, o + 16);
            if (lane < 8) {
#pragma unroll
                for (int c = 0; c < 32; c += 4)
                    *reinterpret_cast<float4 *>(T0 + lane * T16_HSTRIDE + c) = make_float4(o[c], o[c + 1], o[c + 2], o[c + 3]);
            }
        }
        fence_before();
        __syncthreads();  // the table is visible; TMEM lanes 0..7 are free again
    }

    // boards path: a thread needs only the request row of ITS position (prefetched one iteration ahead)
    const T16ReqSpec spec = t16_req_spec(in_tile ? p : 0);
    T16Req cur{};
    if constexpr (BOARDS) cur = t16_req_load(nn_in + min(pair * 3 + j, rows - 1), spec);
    int pos_iter = 0;
    for (int tr = pair; tr < n_triples; tr += n_pairs, ++pos_iter) {
        [[maybe_unused]] const bool dbg_on = blockIdx.x == 0 && pos_iter == 1;
        const int row = tr * 3 + j;                  // this thread's position (global row of the batch)
        const bool real = in_tile && row < rows;     // 13 padding lanes per pair; the last triple may be partial
        T16_STAMP(0);
        float x[64];
        [[maybe_unused]] uint32_t combo = 0;
        if constexpr (!BOARDS) {
            // ---- general float images (AgentModel::evaluate_pv takes any tensor): the reference's 243-float slot read as [81][3] ----
            if (t < 243) {
                IMG[t] = images[(size_t)min(tr * 3 + 0, rows - 1) * 243 + t];
                IMG[243 + t] = images[(size_t)min(tr * 3 + 1, rows - 1) * 243 + t];
                IMG[486 + t] = images[(size_t)min(tr * 3 + 2, rows - 1) * 243 + t];
            }
            __syncthreads();
            const int pc = real ? p : 0;  // padded rows recompute pixel 0 (harmless, never stored)
            const float *im = IMG + (real ? j : 0) * 243;
            const float v0 = im[3 * pc], v1 = im[3 * pc + 1], v2 = im[3 * pc + 2];
            T16_HALF(t16_stem<0>(P, v0, v1, v2, x), t16_stem<1>(P, v0, v1, v2, x));
#pragma unroll
            for (int c = 0; c < 4; ++c) t16_store_group(tlane + TC_X + (uint32_t)t16_chan(half, c * 16), x + c * 16);
        } else {
            // ---- packed boards: the stem of this pixel is a table row ----
            // (block 0's conv0 is a table too, so the packed operand words of the stem row are not needed here: only the
            // fp32 residual row)
            combo = t16_req_combo(cur, spec);
            // prefetch the next triple's request row: its global-load latency hides behind this whole iteration
            if (tr + n_pairs < n_triples) cur = t16_req_load(nn_in + min((tr + n_pairs) * 3 + j, rows - 1), spec);
            const float4 *tx = reinterpret_cast<const float4 *>(T32 + combo * T16_TABSTRIDE + half * 32);
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const float4 v = tx[c + (c >= 8 ? 8 : 0)];  // x[32..63] are channels 64 + 32 half ..
                x[4 * c + 0] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
            }
        }
        if constexpr (!BOARDS) tmem_wait_st();
        T16_STAMP(1);

        // (rolled on purpose: unrolled three times the constant-bank offsets become immediates, but 9.4k instructions of code run no faster)
#pragma unroll 1
        for (int r = 0; r < 3; ++r, ++g) {
            const Tower16Block &B = P.blk[r];
            const uint32_t wb = sbase + S16_W + (g & 1u) * W16_BYTES;
            // ================= conv0: 1x1 128 -> 32 (A = X in TMEM) =================
            if (r == 0 && lane == 0) bulk_wait_read0();  // the write-out's TMA stores have read their staging tiles: the weight prefetch below may overwrite them
            fence_before();
            __syncthreads();
            const bool table0 = BOARDS && r == 0;  // conv0 + epilogue 1 of this block are a table row
            if (table0) {
                if (warp == 3 && lane == 0) {
                    issue_weights(g + 1);
                    mbar_expect_tx(bar_band, T16_BAND_BYTES);
                }
            } else {
                if (warp == 0) {
                    if (elect_one()) {
                        fence_after();
                        mbar_wait(bar_w0 + 8 * (g & 1u), (g >> 1) & 1u);
                        t16_issue_conv0(tmem_base, wb, sbase + S16_ZERO);
                        umma_commit(bar_mma);
                    }
                } else if (lane == 0) {
                    fence_after();
                    if (warp == 3) {
                        issue_weights(g + 1);  // the other buffer's last reader (block g-1, or the write-out) has completed
                        mbar_expect_tx(bar_band, T16_BAND_BYTES);  // arm this block's band phase
                    }
                    umma_commit(bar_mma);
                }
                T16_WAIT_MMA(bar_mma, mma_uses & 1u);
                ++mma_uses;
                fence_after();
            }
            T16_STAMP(2 + r * 8 + 0);
            // epilogue 1: + b0, lrelu -> fp32 tile for the depthwise stencil (this thread: 16 channels of its pixel)
            {
                float d[16], o[16];
                if (table0) {
                    const float4 *t0 = reinterpret_cast<const float4 *>(T0 + combo * T16_HSTRIDE + half * 16);
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 v = t0[c];
                        o[4 * c + 0] = v.x; o[4 * c + 1] = v.y; o[4 * c + 2] = v.z; o[4 * c + 3] = v.w;
                    }
                } else {
                    tmem_ld16(tlane + TC_ACC + half * 16, d);
                    tmem_wait_ld();
                    t16_lrelu_scaled16(B.inv[0], d, o);
                }
                if (in_tile) {
                    float *hrow = H0 + (slot * kCells + p) * T16_HSTRIDE + half * 16;
#pragma unroll
                    for (int c = 0; c < 16; c += 4) *reinterpret_cast<float4 *>(hrow + c) = make_float4(o[c], o[c + 1], o[c + 2], o[c + 3]);
                }
                if (band) {  // the peer keeps this position in its slot 1 - peer_rank = rank
                    mbar_wait(bar_free, (g & 1u) ^ 1u);  // the peer has finished the previous block's stencil
                    const uint32_t ra = peer_h0 + (uint32_t)((((int)rank * kCells + p) * T16_HSTRIDE + half * 16) * 4);
#pragma unroll
                    for (int c = 0; c < 16; c += 4)
                        asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
                                     ::"r"(ra + c * 4), "f"(o[c]), "f"(o[c + 1]), "f"(o[c + 2]), "f"(o[c + 3]), "r"(peer_band) : "memory");
                }
            }
            [[maybe_unused]] float2 wdw[9];
            if constexpr (T16_ROWS) {  // this thread's nine depthwise weight pairs (L1-resident after the first iteration; the latency hides behind the band wait)
                const float2 *wp = reinterpret_cast<const float2 *>(pimg + P16_BLK0 + r * P16_BLK + P16_DW) + cp;
#pragma unroll
                for (int k = 0; k < 9; ++k) wdw[k] = __ldg(wp + k * 16);
                // block 0 of the boards path never waited for its weight image (conv0 is a table): the A tile below overlays W0
                if (BOARDS && r == 0 && warp == 7) mbar_wait(bar_w0 + 8 * (g & 1u), (g >> 1) & 1u);
            }
            T16_WAIT(bar_band, g & 1u);      // the band mirrored by the peer has arrived, and (CTA barrier) this CTA's rows are in the tile
            T16_STAMP(2 + r * 8 + 1);
            // conv1 depthwise 3x3 -> A operand of the pointwise conv
            if constexpr (T16_ROWS) {
                if (has_unit) {
                    const uint32_t mid = sbase + S16_H + (uint32_t)((((uj - (int)rank) * kCells + urow * kSide) * T16_HSTRIDE + cp * 2) * 4);
                    const uint32_t zero = sbase + S16_ZERO + (uint32_t)(cp * 8);
                    const uint32_t up = urow > 0 ? mid - kSide * T16_HSTRIDE * 4 : zero, dn = urow < kSide - 1 ? mid + kSide * T16_HSTRIDE * 4 : zero;
                    const int r0 = uj * kCells + urow * kSide - (int)rank * 128;
                    t16_row_stencil(up, mid, dn, wdw, (uint32_t)((int)(wb + (cp >> 2) * T16_A_CHUNK + (cp & 3) * 4) + r0 * 16), r0);
                }
                fence_proxy_async_smem();  // the A tile was written through the generic proxy; conv1 reads it through the async proxy
            } else {
                float a[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) a[c] = 0.0f;
                if (real) {
                    const float *Hpos = H0 + slot * kCells * T16_HSTRIDE;
                    const int y = p / kSide, xx0 = p - y * kSide;
                    T16_HALF(t16_stencil<0>(B, Hpos, y, xx0, a), t16_stencil<1>(B, Hpos, y, xx0, a));
                }
                t16_store_group(tlane + TC_H + (uint32_t)(half * 16), a);
                tmem_wait_st();
            }
            T16_STAMP(2 + r * 8 + 2);
            // ================= conv1 pointwise: 1x1 32 -> 32 (A = H in TMEM) =================
            fence_before();
            __syncthreads();  // also: every thread's stencil reads of the tile are complete
            if (warp == 0) {
                if (elect_one()) {
                    fence_after();
                    if constexpr (BOARDS) mbar_wait(bar_w0 + 8 * (g & 1u), (g >> 1) & 1u);  // block 0 skipped conv0's wait
                    const uint64_t bhi = desc_sw128(wb + W16_PW), blo = bhi + 4u;
                    const uint32_t dcol = tmem_base + TC_ACC;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        if constexpr (T16_ROWS) {  // A from shared memory: hi chunks 2 ks, 2 ks + 1; lo chunks 4 + 2 ks, 5 + 2 ks
                            const uint64_t ahi = desc_nosw(wb + (uint32_t)(2 * ks * T16_A_CHUNK), T16_A_CHUNK, 128u);
                            const uint64_t alo = desc_nosw(wb + (uint32_t)((4 + 2 * ks) * T16_A_CHUNK), T16_A_CHUNK, 128u);
                            umma_f16_ss<1>(dcol, alo, bhi + (uint64_t)(2 * ks), T16_IDESC_N32, ks != 0);
                            umma_f16_ss<1>(dcol, ahi, blo + (uint64_t)(2 * ks), T16_IDESC_N32, 1u);
                            umma_f16_ss<1>(dcol, ahi, bhi + (uint64_t)(2 * ks), T16_IDESC_N32, 1u);
                        } else {
                            const uint32_t ahi = tmem_base + TC_H + 16u * ks;
                            umma_f16_ts(dcol, ahi + 8u, bhi + (uint64_t)(2 * ks), T16_IDESC_N32, ks != 0);
                            umma_f16_ts(dcol, ahi, blo + (uint64_t)(2 * ks), T16_IDESC_N32, 1u);
                            umma_f16_ts(dcol, ahi, bhi + (uint64_t)(2 * ks), T16_IDESC_N32, 1u);
                        }
                    }
                    umma_f16_ts(dcol, tmem_base + TC_ONE, desc_nosw(wb + W16_B1T, sbase + S16_ZERO - (wb + W16_B1T), 128u), T16_IDESC_N32, 1u);  // + b1
                    umma_commit(bar_mma);
                }
            } else if (lane == 0) {
                fence_after();
                if (warp == 3) mbar_arrive_cluster_relaxed(peer_free);  // the peer may overwrite this CTA's mirrored band (all stencil loads were consumed before the barrier above)
                umma_commit(bar_mma);
            }
            T16_WAIT_MMA(bar_mma, mma_uses & 1u);
            ++mma_uses;
            fence_after();
            T16_STAMP(2 + r * 8 + 3);
            {   // epilogue 2: + b1, lrelu -> A operand of conv2
                float d[16], o[16];
                tmem_ld16(tlane + TC_ACC + half * 16, d);
                tmem_wait_ld();
                t16_lrelu_scaled16(B.inv[1], d, o);
                t16_store_group(tlane + TC_H + (uint32_t)(half * 16), o);
            }
            tmem_wait_st();
            T16_STAMP(2 + r * 8 + 4);
            // ================= conv2: 1x1 32 -> 128 (A = H in TMEM), + x, lrelu =================
            fence_before();
            __syncthreads();
            if (warp == 0) {  // N = 128 MMAs are tensor-bound (64 clk each): one chain
                if (elect_one()) {
                    fence_after();
                    const uint64_t bhi0 = desc_sw128(wb + W16_W2);
                    if constexpr (T16_SPLIT2) {
                        // two N = 64 halves (output channels [0,64) then [64,128): 64 rows of W2^T = 8 KB, 64 rows of the bias tile = 1 KB),
                        // each with its own completion barrier: epilogue 3's first pass needs only the first
#pragma unroll
                        for (int nh = 0; nh < 2; ++nh) {
                            const uint32_t dcol = tmem_base + TC_D3 + 64u * nh;
#pragma unroll
                            for (int ks = 0; ks < 2; ++ks) {
                                const uint64_t bhi = bhi0 + (uint64_t)(nh * 512 + ks * 2), blo = bhi0 + (uint64_t)(nh * 512 + 4 + ks * 2);
                                const uint32_t ahi = tmem_base + TC_H + 16u * ks;
                                umma_f16_ts(dcol, ahi + 8u, bhi, T16_IDESC_N64, ks != 0);
                                umma_f16_ts(dcol, ahi, blo, T16_IDESC_N64, 1u);
                                umma_f16_ts(dcol, ahi, bhi, T16_IDESC_N64, 1u);
                            }
                            const uint32_t bt = wb + W16_B2T + 1024u * nh;
                            umma_f16_ts(dcol, tmem_base + TC_ONE, desc_nosw(bt, sbase + S16_ZERO - bt, 128u), T16_IDESC_N64, 1u);  // + b2 * 2^s
                            umma_commit(nh ? bar_mma2 : bar_mma);
                        }
                    } else {
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            const uint64_t bhi = bhi0 + (uint64_t)(ks * 2), blo = bhi0 + (uint64_t)(4 + ks * 2);
                            const uint32_t ahi = tmem_base + TC_H + 16u * ks;
                            umma_f16_ts(tmem_base + TC_D3, ahi + 8u, bhi, T16_IDESC_N128, ks != 0);
                            umma_f16_ts(tmem_base + TC_D3, ahi, blo, T16_IDESC_N128, 1u);
                            umma_f16_ts(tmem_base + TC_D3, ahi, bhi, T16_IDESC_N128, 1u);
                        }
                        // + b2 * 2^s: constant A group x bias tile (k-chunk 0 = the tile, k-chunk 1 = the shared zero block)
                        umma_f16_ts(tmem_base + TC_D3, tmem_base + TC_ONE, desc_nosw(wb + W16_B2T, sbase + S16_ZERO - (wb + W16_B2T), 128u),
                                    T16_IDESC_N128, 1u);
                        umma_commit(bar_mma);
                    }
                }
            } else if (lane == 0) {
                fence_after();
                umma_commit(bar_mma);
            }
            T16_WAIT_MMA(bar_mma, mma_uses & 1u);
            ++mma_uses;
            fence_after();
            T16_STAMP(2 + r * 8 + 5);
            // epilogue 3: x = lrelu(conv2 + b2 + x); the next block's A operand is written in place over D3
#pragma unroll
            for (int c2 = 0; c2 < 4; c2 += 2) {
                float d[32];
                const int ch0 = t16_chan(half, c2 * 16);  // 32 half (first pass), 64 + 32 half (second pass)
                if constexpr (T16_SPLIT2) {
                    if (c2) {  // the second half of conv2 (columns [64,128)) has its own barrier: complete long before this point
                        mbar_wait(bar_mma2, g & 1u);
                        fence_after();
                    }
                }
                tmem_ld16(tlane + TC_D3 + ch0, d);
                tmem_ld16(tlane + TC_D3 + ch0 + 16, d + 16);
                tmem_wait_ld();
                T16_HALF(t16_residual32<0>(B, c2 * 16, d, x), t16_residual32<1>(B, c2 * 16, d, x));
                if (r < 2) {
                    t16_store_group(tlane + TC_X + (uint32_t)ch0, x + c2 * 16);
                    t16_store_group(tlane + TC_X + (uint32_t)(ch0 + 16), x + c2 * 16 + 16);
                } else {
                    // ---- flatten NHWC (network.rs:127-137): the tower's output leaves as fp16 hi / lo, 32 channels per
                    // pass.  This block's weight buffer is idle now (conv2 has completed) and holds the staging tiles;
                    // the first pass's TMA reads overlap the second half of this epilogue.
                    const uint32_t tile = wb + (uint32_t)warp * 4608u;
                    if (c2) {
                        if (lane == 0) bulk_wait_read0();
                        __syncwarp();
                    }
                    t16_store_pass(tile, lane, x + c2 * 16, &map_hi, &map_lo, ch0, (int)rank * 128 + q * 32, tr);
                }
            }
            tmem_wait_st();
            T16_STAMP(2 + r * 8 + 6);
        }
        T16_STAMP(30);
        T16_STAMP(31);
    }
    // (timestamps: 0 start, 1 stem done, then per block: conv0 done, E1+sync, dw stored, conv1 done, E2 stored, conv2 done, E3 stored)
    // drain the weight prefetch that was issued one block ahead, then release TMEM
    if (t == 0) mbar_wait(bar_w0 + 8 * (g & 1u), (g >> 1) & 1u);
    if (lane == 0) bulk_wait_all0();  // this warp's TMA stores are complete
    fence_before();
    __syncthreads();
    cluster_sync_all();  // no mirrored store or remote arrival is in flight once both CTAs are here
    if (warp == 1) {
        fence_after();
        tmem_dealloc<1>(tmem_base, T16_TMEM_COLS);
    }
}

// Build the per-block B-operand images (K-major SWIZZLE_128B, scaled fp16 hi/lo) and the fp32 parameter image.
// byte offset of (row n, byte b in [0,128)) inside a SWIZZLE_128B K-major tile
__device__ __forceinline__ uint32_t swz128b(int n, int b) {
    return (uint32_t)((n >> 3) * 1024 + (n & 7) * 128 + ((((b >> 4) ^ (n & 7)) & 7) << 4) + (b & 15));
}
struct Tower16PackArgs {
    const float *conv_w, *conv_b;
    const float *w0[3], *b0[3], *dw[3], *pw[3], *b1[3], *w2[3], *b2[3];
};
__global__ void k_tower16_absmax(Tower16PackArgs a, uint32_t *absmax /*[18]: weights [9], then their biases [9]*/) {
    const int which = blockIdx.x % 9;  // 3 * r + {0: w0, 1: pw, 2: w2}
    const bool bias = blockIdx.x >= 9;
    const int r = which / 3, m = which % 3;
    const float *w = bias ? (m == 0 ? a.b0[r] : (m == 1 ? a.b1[r] : a.b2[r])) : (m == 0 ? a.w0[r] : (m == 1 ? a.pw[r] : a.w2[r]));
    const int n = bias ? (m == 2 ? 128 : 32) : (m == 1 ? 1024 : 4096);
    absmax += bias ? 9 : 0;
    uint32_t mx = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) mx = max(mx, __float_as_uint(w[i]) & 0x7FFFFFFFu);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(absmax + which, mx);
}
__device__ __forceinline__ void put_split(uint8_t *img, uint32_t off_hi, uint32_t off_lo, float v) {
    const __half h = __float2half_rn(v);
    *reinterpret_cast<__half *>(img + off_hi) = h;
    *reinterpret_cast<__half *>(img + off_lo) = __float2half_rn(v - __half2float(h));
}
__global__ void k_tower16_pack(Tower16PackArgs a, const uint32_t *absmax, uint8_t *wimg, float *pimg) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;
    for (int r = 0; r < 3; ++r) {
        uint8_t *img = wimg + (size_t)r * W16_BYTES;
        // power-of-two scale of a weight tensor, limited so that its bias tile (b * 2^s / T16_BIAS_ONE) stays below 2^14 too:
        // a network with tiny weights and large biases gets less up-scaling instead of an overflowing bias operand
        auto scale_of = [&](int which) {
            float sc = f16_split_scale(absmax[which]);
            const float bmax = __uint_as_float(absmax[9 + which]);
            while (bmax * sc * (1.0f / T16_BIAS_ONE) >= 16384.0f && sc > 1.0f) sc *= 0.5f;
            return sc;
        };
        const float s0 = scale_of(3 * r + 0), s1 = scale_of(3 * r + 1), s2 = scale_of(3 * r + 2);
        for (int i = tid; i < 128 * 32; i += nth) {  // W0[k][n]: k = cin 0..127, n = cout 0..31
            const int k = i >> 5, n = i & 31;
            const uint32_t off = (uint32_t)(k >> 6) * 4096u + swz128b(n, (k & 63) * 2);
            put_split(img, W16_W0HI + off, W16_W0LO + off, a.w0[r][k * 32 + n] * s0);
        }
        for (int i = tid; i < 32 * 32; i += nth) {  // PW[k][n]
            const int k = i >> 5, n = i & 31;
            put_split(img, W16_PW + swz128b(n, k * 2), W16_PW + swz128b(n, 64 + k * 2), a.pw[r][k * 32 + n] * s1);
        }
        for (int i = tid; i < 32 * 128; i += nth) {  // W2[k][n]: k = cin 0..31, n = cout 0..127
            const int k = i >> 7, n = i & 127;
            put_split(img, W16_W2 + swz128b(n, k * 2), W16_W2 + swz128b(n, 64 + k * 2), a.w2[r][k * 128 + n] * s2);
        }
        for (int n = tid; n < 32; n += nth) {   // bias tiles of conv0 / conv1: [32 n][8 k]
            const uint32_t off = (uint32_t)(n >> 3) * 128u + (uint32_t)(n & 7) * 16u;
            put_split(img, W16_B0T + off, W16_B0T + off + 2u, a.b0[r][n] * s0 * (1.0f / T16_BIAS_ONE));
            put_split(img, W16_B1T + off, W16_B1T + off + 2u, a.b1[r][n] * s1 * (1.0f / T16_BIAS_ONE));
        }
        for (int n = tid; n < 128; n += nth) {  // bias tile of conv2: [128 n][8 k] no-swizzle core matrices, k = 0 / 1 = hi / lo
            const uint32_t off = (uint32_t)W16_B2T + (uint32_t)(n >> 3) * 128u + (uint32_t)(n & 7) * 16u;
            put_split(img, off, off + 2u, a.b2[r][n] * s2 * (1.0f / T16_BIAS_ONE));
        }
        float *pb = pimg + P16_BLK0 + r * P16_BLK;
        for (int i = tid; i < 32; i += nth) {
            pb[P16_B0 + i] = a.b0[r][i];
            pb[P16_B1 + i] = a.b1[r][i];
        }
        for (int i = tid; i < 288; i += nth) pb[P16_DW + i] = a.dw[r][i];
        for (int i = tid; i < 128; i += nth) pb[P16_B2 + i] = a.b2[r][i];
        if (tid == 0) {
            pb[P16_INV + 0] = 1.0f / s0;
            pb[P16_INV + 1] = 1.0f / s1;
            pb[P16_INV + 2] = 1.0f / s2;
            pb[P16_INV + 3] = 0.0f;
        }
    }
    for (int i = tid; i < 384; i += nth) pimg[P16_WSTEM + i] = a.conv_w[i];
    for (int i = tid; i < 128; i += nth) pimg[P16_BSTEM + i] = a.conv_b[i];
}

bool tower16_prepare_weights(omk_ctx *c) {
    NetWeights &w = *c->model;
    if (!w.tower16_wimg) {
        TowerImages t;
        if (t.tower16_wimg.alloc(3 * W16_BYTES) != cudaSuccess || t.tower16_pimg.alloc(P16_FLOATS) != cudaSuccess ||
            t.tower16_absmax.alloc(18) != cudaSuccess)
            return false;
        static_cast<TowerImages &>(w) = std::move(t);
    }
    Tower16PackArgs a;
    a.conv_w = w.t[0];
    a.conv_b = w.t[1];
    for (int r = 0; r < 3; ++r) {
        const int b = 2 + 7 * r;
        a.w0[r] = w.t[b + 0]; a.b0[r] = w.t[b + 1]; a.dw[r] = w.t[b + 2]; a.pw[r] = w.t[b + 3];
        a.b1[r] = w.t[b + 4]; a.w2[r] = w.t[b + 5]; a.b2[r] = w.t[b + 6];
    }
    cudaMemsetAsync(w.tower16_absmax, 0, sizeof(uint32_t) * 18, c->stream);
    cudaMemsetAsync(w.tower16_wimg, 0, 3 * W16_BYTES, c->stream);
    k_tower16_absmax<<<18, 256, 0, c->stream>>>(a, w.tower16_absmax);
    k_tower16_pack<<<16, 256, 0, c->stream>>>(a, w.tower16_absmax, w.tower16_wimg, w.tower16_pimg);
    c->launches += 2;
    // the fp32 parameter image is passed to k_tower16 by value (constant bank): keep a host copy
    w.tower16_params_host.resize(sizeof(Tower16Params));
    if (cudaMemcpyAsync(w.tower16_params_host.data(), w.tower16_pimg, sizeof(Tower16Params), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return false;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return false;
    return true;
}

void tower16_read_timing(long long *out64) { cudaMemcpyFromSymbol(out64, g_t16_dbg, sizeof(long long) * 64); }

// resident CTA pairs the device can hold (two CTAs per SM when shared memory, registers and TMEM allow)
static int tower16_max_pairs(omk_ctx *c) {
    if (c->tower16_pairs > 0) return c->tower16_pairs;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * 2 * c->n_sms);
    cfg.blockDim = dim3(T16_THREADS);
    cfg.dynamicSmemBytes = T16_SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // Two CTAs per SM: 2 x (107 KB, 256 x 128 registers, 256 TMEM columns) fit an SM exactly.  The occupancy API answers
    // one block per SM for this kernel (measured) while the hardware co-schedules two (tower 1.29 -> 0.87 ms with
    // n_sms pairs instead of n_sms / 2), so the grid is sized from the SM count; surplus CTAs would simply queue.
    int n = c->n_sms;
    int api = 0;
    if (cudaOccupancyMaxActiveClusters(&api, k_tower16<false, true>, &cfg) != cudaSuccess) cudaGetLastError();
    if (getenv("OMK_DEBUG")) {
        int per_sm = -1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tower16<false, true>, T16_THREADS, T16_SMEM_BYTES);
        cudaFuncAttributes fa{};
        cudaFuncGetAttributes(&fa, k_tower16<false, true>);
        fprintf(stderr, "omok_b200: k_tower16 CTA pairs: %d (%d SMs); occupancy API: %d clusters, %d blocks/SM; regs %d, static smem %zu, max dyn smem %d, carveout %d\n",
                n, c->n_sms, api, per_sm, fa.numRegs, fa.sharedSizeBytes, fa.maxDynamicSharedSizeBytes, fa.preferredShmemCarveout);
    }
    if (const char *e = getenv("OMK_TOWER_PAIRS")) n = atoi(e) > 0 ? atoi(e) : n;
    c->tower16_pairs = n;
    return n;
}

bool launch_tower_f16(omk_ctx *c, const float *images_dev, int rows_bound) {
    static const bool stamps = getenv("OMK_TOWER_STAMPS") && atoi(getenv("OMK_TOWER_STAMPS")) != 0;
    const bool boards = images_dev == nullptr;
    auto kern = stamps ? (boards ? k_tower16<true, true> : k_tower16<true, false>) : (boards ? k_tower16<false, true> : k_tower16<false, false>);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T16_SMEM_BYTES);
    // two 107 KB CTAs per SM need the full shared-memory carve-out; the default heuristic sizes it for one block
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    const int triples = (rows_bound + 2) / 3;
    const int max_pairs = tower16_max_pairs(c);
    const int pairs = triples < max_pairs ? triples : max_pairs;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(T16_THREADS);
    cfg.dynamicSmemBytes = T16_SMEM_BYTES;
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const NetWeights &m = *c->model;
    const uint8_t *wimg = m.tower16_wimg;
    if (m.tower16_params_host.empty()) return false;
    const Tower16Params &params = *reinterpret_cast<const Tower16Params *>(m.tower16_params_host.data());
    const NNIn *nn_in = c->ws.nn_in;
    const uint32_t *n_req = c->ws.n_req;
    const ActMaps &maps = c->ws.maps;  // the write-out over this workspace's act0 arrays
    const float *pimg = m.tower16_pimg;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, wimg, params, nn_in, images_dev, n_req, rows_bound, maps.tower_st_hi,
                                             maps.tower_st_lo, pimg);
    if (e != cudaSuccess) fprintf(stderr, "omok_b200: cudaLaunchKernelEx(k_tower16): %s\n", cudaGetErrorString(e));
    c->launches++;
    return e == cudaSuccess;
}

}  // namespace omk
