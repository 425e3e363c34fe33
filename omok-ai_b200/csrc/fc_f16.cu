// fc_f16.cu -- K3 tensor-core path for the fully connected layers fc0 (10368 -> 512, 67 % of the network's flops)
// and fc1 (512 -> 512), fp16-split ("3 x FP16") edition.
//
//   C[M x 512] = lrelu( A[M x K] . W[K x 512] + b )        (alpha-zero/src/network.rs:139-163)
//
// fp32-class accuracy on the 5th-gen tensor cores at the FP16 rate: every operand is split x = hi + lo with
// hi = fp16(x) and lo = fp16(x - hi) (22 significant bits; weights are pre-scaled by a power of two so that
// their low parts stay in fp16's normal range) and each k-step issues three tcgen05.mma kind::f16 into one
// TMEM accumulator:    lo.hi + hi.lo + hi.hi     (the dropped lo.lo term is ~2^-22 relative).
// Measured on the CPU (tests/tools/emulate_split.py): priors within 9e-5 of fp64, the same as plain fp32; one-pass
// TF32 misses the 1e-3 bar by 50x and a bf16 split by 1.2x.  Against the 3 x TF32 kernels this replaced (git history:
// fc0_tc.cu) every MMA carries twice the K, operand bytes halve, and the MMA count halves.
//
// The tensor-core accumulator truncates (measured on the TF32 path: 86 % of outputs biased toward zero), so K is
// accumulated in TMEM only over chunks of CHUNK k-blocks; each chunk is drained into fp32 registers with
// round-to-nearest adds while the tensor cores fill the other TMEM buffer.
//
// PAIR = true  (fc0): a CTA pair (2x1 cluster) owns a 256 x 256 tile: each CTA TMA-loads its own 128 rows of A
//                     and HALF of the B tile, tcgen05.mma.cta_group::2 reads both CTAs' shared memory; 3-stage
//                     ring of 64 KB stages; the leader CTA issues, commits multicast to both CTAs.
// PAIR = false (fc1): one CTA per 128 x 256 tile, 2-stage ring of 96 KB stages.
// Warp roles: 0 = TMA producer, 1 = TMEM allocator + MMA issuer, 2..9 = drain / epilogue (two per lane quadrant).
#include <cstdio>
#include <cstdlib>
#include <cuda.h>

#include "omk_internal.h"
#include "tc_ptx.cuh"

namespace omk {

using namespace tc;

constexpr int F_BM = 128, F_BN = 256, F_BK = 64;  // BK fp16 elements = one 128-byte swizzle row
constexpr int F_N = 512;
constexpr int F_K0 = 10368, F_K1 = 512;
constexpr int F_A_BYTES = F_BM * F_BK * 2;        // 16 KB
// k-blocks accumulated in tensor memory between two drains into fp32 registers.  The tensor-core accumulator truncates,
// so a layer's error grows with the chunk length (profiles/r02_net_error_study.md: 20 000 positions, 3 weight seeds):
//   fc1 / heads  8 -> 1 k-block: max relative prior error 4.6e-4 -> 2.1e-4, +0.001 ms per 16 k rows: the default;
//   fc0          9 -> 3 k-blocks: 2.1e-4 -> 1.6e-4, fc0 +0.8 % on 16 k-row batches, but three times the partial sums of the
//                split-K path (small batches: 8 rows 22 -> 31 us, 1024 rows 51 -> 96 us): OPT-IN at run time
//                (omk_debug_set_fc0_chunk(ctx, 3) / env OMK_FC0_CHUNK=3); both chunkings keep a row's result independent
//                of the batch size and of the path (pair / split-K) its batch takes.
#ifndef OMK_F_CHUNK1
#define OMK_F_CHUNK1 1
#endif
#ifndef OMK_F_CHUNKH
#define OMK_F_CHUNKH 1
#endif
constexpr int F_SPLITK_KB = 9;                    // k-blocks per CTA of the split-K fc0 (small batches)
constexpr int F_CHUNK0 = 9, F_CHUNK0_FINE = 3;    // fc0: 162 k-blocks = 18 x 9 (default) or 54 x 3 (fc0_chunk == 3)
constexpr int F_CHUNK1 = OMK_F_CHUNK1;            // fc1: 8 k-blocks
constexpr int F_CHUNKH = OMK_F_CHUNKH;            // heads: 8 k-blocks
constexpr int kSplitKMaxRows = 2048;              // fc0 batches up to here take the split-K path (36 CTAs per 128 rows): 95 vs 152 us at 2048 rows, 181 vs 158 us at 4096

// TAIL BALANCING of the CTA-pair fc0 (bit-exact).  A launch of T pair-tiles on P resident CTA pairs runs whole waves; in
// the last, partial wave (R = T mod P tiles) the other H = P - R pairs would idle (the search lanes launch 64 tiles for 74
// pairs).  Instead the R "main" pairs accumulate only the first m chunks of their tile, and the H "helper" pairs compute the
// last `tail` = NCHUNK - m chunks of every main tile as stand-alone chunk sums, stored raw to a scratch buffer; a main pair
// then adds its tile's tail chunks IN ORDER after its own m -- the same partial sums in the same order as the unsplit loop,
// so every row keeps its bits (tests/test_net_gpu.py::test_batch_invariance, ::test_fc0_tail_balancing) -- and runs the usual
// epilogue.  A helper's units form one flat k-block stream (no pipeline refill between units).  Helpers have the lowest
// block indices of the wave, so they are resident before the mains that wait for them (per-tile release / acquire counters
// in global memory, bounded spins that trap instead of hanging).
struct FcBal {
    int full;         // clusters [0, full): whole tiles (earlier, complete waves)
    int helpers;      // clusters [full, full + helpers): helper pairs
    int m, tail;      // a main tile: chunks [0, m) by its own pair, [m, m + tail) by helpers
    int mains;        // main tiles (clusters [full + helpers, full + helpers + mains), tile = cluster - helpers)
    float4 *partial;  // [mains * tail units][2 CTAs][8 drain warps][32 float4 groups][32 lanes]
    uint32_t *flags;  // [2][mains]: arrived helper warps per main tile, main warps done with the tile
};
constexpr int F_BAL_TAIL_MAX = 4;
constexpr size_t F_BAL_UNIT_F4 = 2 * 8 * 32 * 32;  // float4 per unit (one 256 x 256 chunk sum)
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <bool PAIR, int BN>
struct FcCfg {
    static constexpr int kStages = PAIR ? 3 : 2;  // (a third 64 KB stage for the 128-column tiles -- heads, narrow split-K fc0 -- measured +-0: same-box A/B)  // 64 KB stages: three fit (heads, the narrow split-K fc0); 96 KB stages: two
    static constexpr int kBRows = PAIR ? BN / 2 : BN;             // B rows loaded by one CTA
    static constexpr int kBBytes = kBRows * F_BK * 2;             // 16 / 32 KB
    static constexpr int kStageBytes = 2 * F_A_BYTES + 2 * kBBytes;  // 64 / 96 KB
    static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 1024;
    static constexpr uint32_t kIdesc = idesc_f16(PAIR ? 256 : 128, BN);
    static constexpr int kDrainWarps = 4 * (BN / 128);            // one warp per lane quadrant and 128-column slab
    static constexpr int kThreads = 64 + 32 * kDrainWarps;
    static constexpr uint32_t kTmemCols = 2 * BN;                 // two accumulator buffers
};

// BN = 256: fc0 / fc1 tiles.  BN = 128 with HEADS: the policy/value heads (512 -> 81 | 1, padded to 128 columns): a drain
// thread owns a whole row of logits, so tanh (value, network.rs:188-202) and softmax (policy, :227-247) finish in registers;
// with LOGITS it stores the row's 82 logits to C [rows][128] instead (policy 0..80, value 81: the layout the CUDA-core heads
// GEMM writes to ws.logits), for the replay score's losses.
// SPLITK (small batches): blockIdx.z selects F_SPLITK_KB k-blocks; the CTA writes the raw fp32 partial sums of each of their chunks
// to C[z][gridDim.y * 128 rows][512] and k_fc0_reduce adds the chunks in order -- the same partial sums in the same order as the
// unsplit kernel, so a row's result stays bit-identical whatever the batch size (recorded-mode parity).
template <int K, int CHUNK, bool PAIR, int BN = 256, bool HEADS = false, bool SPLITK = false, bool LOGITS = false>
__global__ void __launch_bounds__((FcCfg<PAIR, BN>::kThreads), 1)
    k_fc16(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
           const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
           const float *__restrict__ bias, const float *__restrict__ inv_scale_p, float *__restrict__ C,
           __half *__restrict__ C_hi, __half *__restrict__ C_lo, const uint32_t *n_req, int max_rows,
           float *__restrict__ P_out = nullptr, float *__restrict__ V_out = nullptr, uint32_t *dev_error = nullptr,
           const FcBal bal = FcBal{}) {
    using Cfg = FcCfg<PAIR, BN>;
    static_assert(!HEADS || (BN == 128 && !PAIR), "the heads epilogue needs a whole logit row per thread");
    constexpr int CG = PAIR ? 2 : 1;
    static_assert(K % F_BK == 0 && (K / F_BK) % CHUNK == 0, "chunking must tile K");
    static_assert(!SPLITK || (!PAIR && !HEADS), "split-K is the one-CTA fc0 variant");
    static_assert(!LOGITS || HEADS, "LOGITS is an epilogue of the heads");
    // split-K: one CTA walks F_SPLITK_KB k-blocks = several chunks, and stores every chunk's partial sums separately
    constexpr int NKB = SPLITK ? F_SPLITK_KB : K / F_BK;      // k-blocks this CTA walks
    static_assert(!SPLITK || (F_SPLITK_KB % CHUNK == 0 && (K / F_BK) % F_SPLITK_KB == 0), "split-K groups must tile K");
    constexpr int NCHUNK = NKB / CHUNK;
    const int kb_base = SPLITK ? (int)blockIdx.z * F_SPLITK_KB : 0;
    extern __shared__ uint8_t smem_raw[];
    const int rows = (int)min(*n_req, (uint32_t)max_rows);
    uint32_t rank = 0;
    int m0, n0;
    // (pair kernel) this cluster's role and its sequence of chunks: whole tile = chunks [0, NCHUNK) of one tile; main = chunks
    // [0, m) of one tile, then the helpers' tail sums; helper = units [u0, u1), unit u = chunk m + u % tail of main tile u / tail
    [[maybe_unused]] int role = 0, n_seq = NCHUNK, u0 = 0;  // role: 0 whole, 1 main, 2 helper
    [[maybe_unused]] int tile = 0;
    if constexpr (PAIR) {
        // tile = pair * 2 + n_tile: the two N tiles of one row pair are neighbours in launch order so that the second reads
        // its A rows from L2, not from DRAM
        rank = cluster_rank();
        const int cid = blockIdx.x >> 1;
        tile = cid;
        if (cid >= bal.full && bal.helpers > 0) {
            if (cid < bal.full + bal.helpers) {
                role = 2;
                const int units = bal.mains * bal.tail, h = cid - bal.full;
                const int per = (units + bal.helpers - 1) / bal.helpers;
                u0 = h * per;
                n_seq = max(0, min(units, u0 + per) - u0);
            } else {
                role = 1;
                tile = cid - bal.helpers;
                n_seq = bal.m;
            }
        }
        const int pair = tile >> 1;
        m0 = pair * 256 + (int)rank * F_BM;
        n0 = (tile & 1) * BN;
        if (role != 2 && pair * 256 >= rows) return;  // uniform for the whole cluster
    } else {
        m0 = blockIdx.y * F_BM;
        n0 = blockIdx.x * BN;
        if (m0 >= rows) return;  // uniform for the whole CTA, before any barrier or TMEM use
    }
    const bool leader = rank == 0;

    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t bars = base + Cfg::kStages * Cfg::kStageBytes;
    const uint32_t full0 = bars, empty0 = bars + 8 * Cfg::kStages, tmem_full0 = bars + 16 * Cfg::kStages,
                   tmem_empty0 = tmem_full0 + 16, tmem_slot = tmem_empty0 + 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        prefetch_map(&map_a_hi);
        prefetch_map(&map_a_lo);
        prefetch_map(&map_b_hi);
        prefetch_map(&map_b_lo);
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(tmem_full0 + 8 * b, 1);
            mbar_init(tmem_empty0 + 8 * b, (PAIR ? 2 : 1) * Cfg::kDrainWarps);  // one arrival per drain warp (of both CTAs)
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<CG>(tmem_slot, Cfg::kTmemCols);
    fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // both CTAs' barriers are initialised before anything crosses the pair
    fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            if constexpr (PAIR) {  // both CTAs load; the transaction bytes of both land on the leader's barrier
                int it = 0;  // flat k-block counter of this cluster (the ring runs through unit boundaries)
                for (int i = 0; i < n_seq; ++i) {
                    int ch = i, mm = m0, nn = n0;
                    if (role == 2) {
                        const int u = u0 + i, tl = bal.full + u / bal.tail;
                        ch = bal.m + u % bal.tail;
                        mm = (tl >> 1) * 256 + (int)rank * F_BM;
                        nn = (tl & 1) * BN;
                        if ((tl >> 1) * 256 >= rows) continue;  // that main pair has left: nobody reads this unit
                    }
                    for (int kc = 0; kc < CHUNK; ++kc, ++it) {
                        const int kb = ch * CHUNK + kc, s = it % Cfg::kStages;
                        const uint32_t ph = (uint32_t)(it / Cfg::kStages) & 1u;
                        mbar_wait(empty0 + 8 * s, ph ^ 1u);
                        const uint32_t st = base + s * Cfg::kStageBytes;
                        const uint32_t lbar = mapa(full0 + 8 * s, 0);
                        if (leader) mbar_expect_tx(full0 + 8 * s, 2 * Cfg::kStageBytes);
                        tma_load_2d_2sm(st, &map_a_hi, lbar, kb * F_BK, mm);
                        tma_load_2d_2sm(st + F_A_BYTES, &map_a_lo, lbar, kb * F_BK, mm);
                        tma_load_2d_2sm(st + 2 * F_A_BYTES, &map_b_hi, lbar, kb * F_BK, nn + (int)rank * 128);
                        tma_load_2d_2sm(st + 2 * F_A_BYTES + Cfg::kBBytes, &map_b_lo, lbar, kb * F_BK, nn + (int)rank * 128);
                    }
                }
            }
            for (int kb = 0; kb < (PAIR ? 0 : NKB); ++kb) {
                const int s = kb % Cfg::kStages;
                const uint32_t ph = (uint32_t)(kb / Cfg::kStages) & 1u;
                mbar_wait(empty0 + 8 * s, ph ^ 1u);
                const uint32_t st = base + s * Cfg::kStageBytes;
                if constexpr (PAIR) {
                } else {
                    const uint32_t bar = full0 + 8 * s;
                    mbar_expect_tx(bar, Cfg::kStageBytes);
                    tma_load_2d(st, &map_a_hi, bar, (kb_base + kb) * F_BK, m0);
                    tma_load_2d(st + F_A_BYTES, &map_a_lo, bar, (kb_base + kb) * F_BK, m0);
                    tma_load_2d(st + 2 * F_A_BYTES, &map_b_hi, bar, (kb_base + kb) * F_BK, n0);
                    tma_load_2d(st + 2 * F_A_BYTES + Cfg::kBBytes, &map_b_lo, bar, (kb_base + kb) * F_BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        if (leader && lane == 0) {  // ===== MMA issuer (the leader CTA of a pair) =====
            for (int i = 0, ci = 0, it = 0; i < n_seq; ++i) {  // ci: chunks issued, it: k-blocks consumed (ring position)
                if constexpr (PAIR) {
                    if (role == 2 && ((bal.full + (u0 + i) / bal.tail) >> 1) * 256 >= rows) continue;  // skipped unit (see the producer)
                }
                const int buf = ci & 1;
                const uint32_t use = (uint32_t)(ci >> 1);
                ++ci;
                mbar_wait(tmem_empty0 + 8 * buf, (use & 1u) ^ 1u);  // drained (passes at once for the first use)
                fence_after();
                const uint32_t tmem_acc = tmem_base + (uint32_t)(buf * BN);
                for (int kc = 0; kc < CHUNK; ++kc, ++it) {
                    const int s = it % Cfg::kStages;
                    const uint32_t ph = (uint32_t)(it / Cfg::kStages) & 1u;
                    mbar_wait(full0 + 8 * s, ph);
                    fence_after();
                    const uint32_t st = base + s * Cfg::kStageBytes;
                    const uint64_t a_hi = desc_sw128(st), a_lo = desc_sw128(st + F_A_BYTES);
                    const uint64_t b_hi = desc_sw128(st + 2 * F_A_BYTES), b_lo = desc_sw128(st + 2 * F_A_BYTES + Cfg::kBBytes);
#pragma unroll
                    for (int k = 0; k < F_BK / 16; ++k) {
                        const uint64_t adv = (uint64_t)((k * 32) >> 4);  // 16 fp16 = 32 bytes per k-step inside the swizzle atom
                        umma_f16_ss<CG>(tmem_acc, a_lo + adv, b_hi + adv, Cfg::kIdesc, (kc | k) != 0 ? 1u : 0u);
                        umma_f16_ss<CG>(tmem_acc, a_hi + adv, b_lo + adv, Cfg::kIdesc, 1u);
                        umma_f16_ss<CG>(tmem_acc, a_hi + adv, b_hi + adv, Cfg::kIdesc, 1u);
                    }
                    if constexpr (PAIR) umma_commit_2sm(empty0 + 8 * s); else umma_commit(empty0 + 8 * s);
                }
                if constexpr (PAIR) umma_commit_2sm(tmem_full0 + 8 * buf); else umma_commit(tmem_full0 + 8 * buf);
            }
        }
    } else {  // ===== drain + epilogue: warps 2..9; lane quadrant = warp % 4, column half = (warp - 2) / 4 =====
        const int q = warp & 3, half = (warp - 2) >> 2;
        float acc[128];
#pragma unroll
        for (int j = 0; j < 128; ++j) acc[j] = 0.0f;
        for (int ch = 0, ci = 0; ch < n_seq; ++ch) {
            [[maybe_unused]] float4 *unit_dst = nullptr;  // helper: where this unit's raw chunk sums go
            [[maybe_unused]] int unit_main = 0;
            if constexpr (PAIR) {
                if (role == 2) {
                    const int u = u0 + ch;
                    unit_main = u / bal.tail;
                    if (((bal.full + unit_main) >> 1) * 256 >= rows) continue;  // skipped unit (see the producer)
                    unit_dst = bal.partial + (((size_t)u * 2 + rank) * 8 + (size_t)(warp - 2)) * 1024 + lane;
                }
            }
            const int buf = ci & 1;
            const uint32_t use = (uint32_t)(ci >> 1);
            ++ci;
            mbar_wait(tmem_full0 + 8 * buf, use & 1u);
            fence_after();
#pragma unroll
            for (int c = 0; c < 128; c += 32) {
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + half * 128 + c), v);
                tmem_wait_ld();
                if (PAIR && role == 2) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) unit_dst[(size_t)((c + j) >> 2) * 32] = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[c + j] += v[j];
                }
            }
            fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_cluster(mapa(tmem_empty0 + 8 * buf, 0)); else mbar_arrive(tmem_empty0 + 8 * buf);
            }
            if constexpr (PAIR) {
                if (role == 2) {  // release this warp's share of the unit to the main pair of the tile
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) atomicAdd(bal.flags + unit_main, 1u);
                }
            }
            if constexpr (SPLITK) {  // raw partial sums of THIS chunk: C[chunk index][row in tile][512]; the accumulator restarts
                const int prow = m0 + q * 32 + lane;
                if (prow < rows) {
                    float *dst = C + ((size_t)((int)blockIdx.z * NCHUNK + ch) * ((size_t)gridDim.y * F_BM) + (size_t)prow) * F_N + n0 + half * 128;
#pragma unroll
                    for (int j = 0; j < 128; j += 4) *reinterpret_cast<float4 *>(dst + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
                }
#pragma unroll
                for (int j = 0; j < 128; ++j) acc[j] = 0.0f;
            }
        }
        if constexpr (PAIR) {
            if (role == 1) {  // the tile's tail chunks, computed by helper pairs: add them in order behind this pair's own m chunks
                const int k = tile - bal.full;
                const uint32_t need = (uint32_t)bal.tail * 16u;  // 8 drain warps x 2 CTAs per unit
                uint32_t spin = 0;
                while (ld_acquire_u32(bal.flags + k) < need) {
                    if (++spin > (1u << 22)) __trap();  // a scheduling assumption broke: fail loudly instead of hanging
                    __nanosleep(64);
                }
                for (int j = 0; j < bal.tail; ++j) {
                    const float4 *src = bal.partial + (((size_t)(k * bal.tail + j) * 2 + rank) * 8 + (size_t)(warp - 2)) * 1024 + lane;
#pragma unroll
                    for (int c4 = 0; c4 < 32; ++c4) {
                        const float4 v = __ldcg(src + (size_t)c4 * 32);
                        acc[4 * c4 + 0] += v.x; acc[4 * c4 + 1] += v.y; acc[4 * c4 + 2] += v.z; acc[4 * c4 + 3] += v.w;
                    }
                }
                __syncwarp();
                if (lane == 0 && atomicAdd(bal.flags + 128 + k, 1u) == 15u) {  // the last of the tile's 16 main warps re-arms the counters
                    atomicExch(bal.flags + k, 0u);
                    atomicExch(bal.flags + 128 + k, 0u);
                }
            }
        }
        const int row = m0 + q * 32 + lane;
        const size_t coff = (size_t)row * F_N + n0 + half * 128;
        const float *brow = bias + n0 + half * 128;
        const float inv_scale = *inv_scale_p;  // undo the power-of-two weight scaling (exact)
        if constexpr (SPLITK) {
            // (the chunks' partial sums were stored in the drain loop)
        } else if constexpr (LOGITS) {
            if (row < rows) {
                // the logits exactly as the branch below forms them before softmax / tanh
                float *lrow = C + (size_t)row * 128;
                bool finite = true;
#pragma unroll
                for (int j = 0; j < 80; j += 4) {
                    const float4 o = make_float4(fmaf(acc[j], inv_scale, brow[j]), fmaf(acc[j + 1], inv_scale, brow[j + 1]),
                                                 fmaf(acc[j + 2], inv_scale, brow[j + 2]), fmaf(acc[j + 3], inv_scale, brow[j + 3]));
                    finite = finite && fabsf(o.x) < INFINITY && fabsf(o.y) < INFINITY && fabsf(o.z) < INFINITY && fabsf(o.w) < INFINITY;
                    *reinterpret_cast<float4 *>(lrow + j) = o;
                }
                const float l80 = fmaf(acc[80], inv_scale, brow[80]), vlogit = fmaf(acc[kCells], inv_scale, brow[kCells]);
                if (!finite || !(fabsf(l80) < INFINITY) || !(fabsf(vlogit) < INFINITY)) atomicOr(dev_error, 2u);
                lrow[80] = l80;
                lrow[kCells] = vlogit;
            }
        } else if constexpr (HEADS) {
            if (row < rows) {
                // logits: columns 0..80 policy, 81 value (k_pack_heads); same softmax / tanh arithmetic as k_heads
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < kCells; ++j) {
                    acc[j] = fmaf(acc[j], inv_scale, brow[j]);
                    mx = fmaxf(mx, acc[j]);
                }
                float sum = 0.0f;
#pragma unroll
                for (int j = 0; j < kCells; ++j) {
                    acc[j] = expf(acc[j] - mx);
                    sum += acc[j];
                }
                const float inv = 1.0f / sum;
                const float vlogit = fmaf(acc[kCells], inv_scale, brow[kCells]);
                // loud failure instead of silent garbage: an fp16 operand overflow upstream shows up here as NaN / Inf
                if (!(sum >= 1.0f && sum < INFINITY) || !(fabsf(vlogit) < INFINITY)) atomicOr(dev_error, 2u);
                float *prow = P_out + (size_t)row * kRow;
#pragma unroll
                for (int j = 0; j < 80; j += 4)
                    *reinterpret_cast<float4 *>(prow + j) = make_float4(acc[j] * inv, acc[j + 1] * inv, acc[j + 2] * inv, acc[j + 3] * inv);
                prow[80] = acc[80] * inv;
                V_out[row] = tanhf(vlogit);
            }
        } else if (row < rows && role != 2) {  // rows past the batch are never stored (the tile may extend past the workspace)
#pragma unroll
            for (int j = 0; j < 128; j += 8) {
                float o[8];
#pragma unroll
                for (int i = 0; i < 8; i += 4) {
                    const float4 b = *reinterpret_cast<const float4 *>(brow + j + i);
                    o[i + 0] = fmaf(acc[j + i + 0], inv_scale, b.x);
                    o[i + 1] = fmaf(acc[j + i + 1], inv_scale, b.y);
                    o[i + 2] = fmaf(acc[j + i + 2], inv_scale, b.z);
                    o[i + 3] = fmaf(acc[j + i + 3], inv_scale, b.w);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = fmaxf(o[i], 0.2f * o[i]);
                if (C) {
                    *reinterpret_cast<float4 *>(C + coff + j) = make_float4(o[0], o[1], o[2], o[3]);
                    *reinterpret_cast<float4 *>(C + coff + j + 4) = make_float4(o[4], o[5], o[6], o[7]);
                }
                if (C_hi) {
                    uint4 h, l;
                    split2_f16(o[0], o[1], h.x, l.x);
                    split2_f16(o[2], o[3], h.y, l.y);
                    split2_f16(o[4], o[5], h.z, l.z);
                    split2_f16(o[6], o[7], h.w, l.w);
                    *reinterpret_cast<uint4 *>(C_hi + coff + j) = h;
                    *reinterpret_cast<uint4 *>(C_lo + coff + j) = l;
                }
            }
        }
    }
    fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // the peer's shared memory and TMEM stay alive until every MMA and drain has finished
    if (warp == 1) {
        fence_after();
        tmem_dealloc<CG>(tmem_base, Cfg::kTmemCols);
    }
}

// split-K tail of fc0 for small batches: chunks added in order (bit-identical to the register accumulation of k_fc16),
// then the same epilogue: * 2^-s + bias, lrelu, fp16 hi/lo split
__global__ void k_fc0_reduce(const float *__restrict__ partial, int nchunks, int ws_rows, const float *__restrict__ bias,
                             const float *__restrict__ inv_scale_p, __half *__restrict__ C_hi, __half *__restrict__ C_lo,
                             const uint32_t *n_req, int max_rows) {
    const int rows = (int)min(*n_req, (uint32_t)max_rows);
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // (row, group of 8 columns)
    const int row = idx >> 6, j = (idx & 63) * 8;
    if (row >= rows) return;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0f;
    // six chunks' loads in flight at a time, added in chunk order (one chunk at a time was a chain of 18 / 54 exposed L2
    // latencies: 8.5 us for a batch of 8 rows)
    for (int z0 = 0; z0 < nchunks; z0 += 6) {
        float4 a[6], b[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int z = min(z0 + i, nchunks - 1);
            const float *p = partial + ((size_t)z * ws_rows + row) * F_N + j;
            a[i] = *reinterpret_cast<const float4 *>(p);
            b[i] = *reinterpret_cast<const float4 *>(p + 4);
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            if (z0 + i >= nchunks) break;
            acc[0] += a[i].x; acc[1] += a[i].y; acc[2] += a[i].z; acc[3] += a[i].w;
            acc[4] += b[i].x; acc[5] += b[i].y; acc[6] += b[i].z; acc[7] += b[i].w;
        }
    }
    const float inv_scale = *inv_scale_p;
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        o[i] = fmaf(acc[i], inv_scale, bias[j + i]);
        o[i] = fmaxf(o[i], 0.2f * o[i]);
    }
    uint4 h, l;
    split2_f16(o[0], o[1], h.x, l.x);
    split2_f16(o[2], o[3], h.y, l.y);
    split2_f16(o[4], o[5], h.z, l.z);
    split2_f16(o[6], o[7], h.w, l.w);
    *reinterpret_cast<uint4 *>(C_hi + (size_t)row * F_N + j) = h;
    *reinterpret_cast<uint4 *>(C_lo + (size_t)row * F_N + j) = l;
}

// max |w| of a tensor as fp32 bits (non-negative floats order like their bit patterns)
__global__ void k_absmax_bits(const float *__restrict__ w, long long n, uint32_t *out) {
    uint32_t m = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = max(m, __float_as_uint(w[i]) & 0x7FFFFFFFu);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// W[K][N] -> K-major transposed fp16 hi / lo parts Wt[N][K] of W * 2^s; writes 2^-s to *inv_scale
__global__ void k_fc16_split_weights(const float *__restrict__ W, const uint32_t *absmax_bits, __half *__restrict__ hi,
                                     __half *__restrict__ lo, float *inv_scale, int K, int N) {
    __shared__ float tile[32][33];
    const float scale = f16_split_scale(*absmax_bits);
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *inv_scale = 1.0f / scale;
    const int k0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int r = ty; r < 32; r += 8) tile[r][tx] = W[(size_t)(k0 + r) * N + n0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const float x = tile[tx][r] * scale;  // W[k0+tx][n0+r]
        const __half h = __float2half_rn(x);
        hi[(size_t)(n0 + r) * K + k0 + tx] = h;
        lo[(size_t)(n0 + r) * K + k0 + tx] = __float2half_rn(x - __half2float(h));
    }
}

// debug / A-B helpers: fp32 activations <-> fp16 hi/lo split (lets either half of the network run on another path)
__global__ void k_f32_to_split16(const float *__restrict__ x, __half *__restrict__ hi, __half *__restrict__ lo, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const __half h = __float2half_rn(x[i]);
        hi[i] = h;
        lo[i] = __float2half_rn(x[i] - __half2float(h));
    }
}
__global__ void k_split16_to_f32(const __half *__restrict__ hi, const __half *__restrict__ lo, float *__restrict__ x, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        x[i] = __half2float(hi[i]) + __half2float(lo[i]);
}
void launch_f32_to_split16(omk_ctx *c, const float *x, __half *hi, __half *lo, long long n) {
    k_f32_to_split16<<<1184, 256, 0, c->stream>>>(x, hi, lo, n);
    c->launches++;
}
void launch_split16_to_f32(omk_ctx *c, const __half *hi, const __half *lo, float *x, long long n) {
    k_split16_to_f32<<<1184, 256, 0, c->stream>>>(hi, lo, x, n);
    c->launches++;
}

typedef CUresult (*PFN_encodeTiled16)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D fp16 [rows][K] row-major, boxes of box_rows x 64 elements (128-byte rows), SWIZZLE_128B
static bool encode_map16(CUtensorMap *map, __half *ptr, uint64_t rows, uint32_t box_rows, int K) {
    static PFN_encodeTiled16 fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return false;
        fn = (PFN_encodeTiled16)p;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)K * sizeof(__half)};
    const cuuint32_t box[2] = {(cuuint32_t)F_BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 3-D fp16 view [triple][243 pixel rows][128 channels] of a tower output array for k_tower16's TMA write-out: boxes of 32
// rows x 32 channels (64 bytes), SWIZZLE_64B; a CTA pair's 13 padding rows (>= 243) fall outside dimension 1 and are clipped
static bool encode_map_tower_store(CUtensorMap *map, __half *ptr, uint64_t rows) {
    static PFN_encodeTiled16 fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return false;
        fn = (PFN_encodeTiled16)p;
    }
    const cuuint64_t dims[3] = {128, 243, (rows + 2) / 3};  // the arrays carry two rows of slack for the last triple
    const cuuint64_t strides[2] = {128 * sizeof(__half), 243 * 128 * sizeof(__half)};
    const cuuint32_t box[3] = {32, 32, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct Fc16State {  // what belongs to the device, shared by both models and both search lanes
    int pair_slots = 0;  // CTA pairs of the fc0 pair kernel the device holds at once (0 = not queried yet)
};
void Fc16StateFree::operator()(Fc16State *s) const { delete s; }

static Fc16State *state16_of(omk_ctx *c) {
    if (!c->fc16_state) c->fc16_state.reset(new Fc16State());
    return c->fc16_state.get();
}

// (re)build the scaled, split, transposed weights of fc0 and fc1; call after the weights change
bool fc16_prepare_weights(omk_ctx *c) {
    NetWeights &w = *c->model;
    if (!w.fc0_wt_h16) {
        FcImages f;
        if (f.fc0_wt_h16.alloc((size_t)F_K0 * F_N) != cudaSuccess || f.fc0_wt_l16.alloc((size_t)F_K0 * F_N) != cudaSuccess ||
            f.fc1_wt_h16.alloc((size_t)F_K1 * F_N) != cudaSuccess || f.fc1_wt_l16.alloc((size_t)F_K1 * F_N) != cudaSuccess ||
            f.heads_wt_h16.alloc((size_t)F_K1 * 128) != cudaSuccess || f.heads_wt_l16.alloc((size_t)F_K1 * 128) != cudaSuccess ||
            f.fc_inv_scale.alloc(3) != cudaSuccess || f.fc_absmax.alloc(3) != cudaSuccess)
            return false;
        static_cast<FcImages &>(w) = std::move(f);
    }
    cudaMemsetAsync(w.fc_absmax, 0, sizeof(uint32_t) * 3, c->stream);
    k_absmax_bits<<<592, 256, 0, c->stream>>>(w.t[23], (long long)F_K0 * F_N, w.fc_absmax);
    k_absmax_bits<<<148, 256, 0, c->stream>>>(w.t[25], (long long)F_K1 * F_N, w.fc_absmax + 1);
    k_absmax_bits<<<64, 256, 0, c->stream>>>(w.heads_w, (long long)F_K1 * 128, w.fc_absmax + 2);  // packed by net_pack_heads
    k_fc16_split_weights<<<dim3(F_K0 / 32, F_N / 32), 256, 0, c->stream>>>(w.t[23], w.fc_absmax, w.fc0_wt_h16, w.fc0_wt_l16,
                                                                           w.fc_inv_scale, F_K0, F_N);
    k_fc16_split_weights<<<dim3(F_K1 / 32, F_N / 32), 256, 0, c->stream>>>(w.t[25], w.fc_absmax + 1, w.fc1_wt_h16, w.fc1_wt_l16,
                                                                           w.fc_inv_scale + 1, F_K1, F_N);
    k_fc16_split_weights<<<dim3(F_K1 / 32, 128 / 32), 256, 0, c->stream>>>(w.heads_w, w.fc_absmax + 2, w.heads_wt_h16, w.heads_wt_l16,
                                                                         w.fc_inv_scale + 2, F_K1, 128);
    c->launches += 6;
    if (!encode_map16(&w.map0_b_hi, w.fc0_wt_h16, F_N, 128, F_K0)) return false;
    if (!encode_map16(&w.map0_b_lo, w.fc0_wt_l16, F_N, 128, F_K0)) return false;
    if (!encode_map16(&w.map0s_b_hi, w.fc0_wt_h16, F_N, F_BN, F_K0)) return false;
    if (!encode_map16(&w.map0s_b_lo, w.fc0_wt_l16, F_N, F_BN, F_K0)) return false;
    if (!encode_map16(&w.map1_b_hi, w.fc1_wt_h16, F_N, F_BN, F_K1)) return false;
    if (!encode_map16(&w.map1_b_lo, w.fc1_wt_l16, F_N, F_BN, F_K1)) return false;
    if (!encode_map16(&w.map2_b_hi, w.heads_wt_h16, 128, 128, F_K1)) return false;
    if (!encode_map16(&w.map2_b_lo, w.heads_wt_l16, 128, 128, F_K1)) return false;
    w.weights_ready = true;
    return true;
}

bool fc16_encode_act_maps(Activations &a) {
    ActMaps &m = a.maps;
    const uint64_t rows = (uint64_t)a.act_rows;
    return encode_map16(&m.map0_a_hi, a.act0_h16, rows, F_BM, F_K0) && encode_map16(&m.map0_a_lo, a.act0_l16, rows, F_BM, F_K0) &&
           encode_map16(&m.map1_a_hi, a.act1_h16, rows, F_BM, F_K1) && encode_map16(&m.map1_a_lo, a.act1_l16, rows, F_BM, F_K1) &&
           encode_map16(&m.map2_a_hi, a.act2_h16, rows, F_BM, F_K1) && encode_map16(&m.map2_a_lo, a.act2_l16, rows, F_BM, F_K1) &&
           encode_map_tower_store(&m.tower_st_hi, a.act0_h16, rows) && encode_map_tower_store(&m.tower_st_lo, a.act0_l16, rows);
}

static bool check_launch(const char *what) {
    const cudaError_t le = cudaPeekAtLastError();
    if (le == cudaSuccess) return true;
    fprintf(stderr, "omok_b200: %s launch failed: %s\n", what, cudaGetErrorString(le));
    return false;
}

// fc0: act0_h16/l16 -> act1_h16/l16 (the A operand of fc1)
bool launch_fc0_f16(omk_ctx *c, int rows_bound) {
    const NetWeights &m = *c->model;
    const ActMaps *am = m.weights_ready ? &c->ws.maps : nullptr;
    if (!am) return false;
    const bool fine = c->fc0_chunk == F_CHUNK0_FINE;
    static const int splitk_env = getenv("OMK_FC0_SPLITK_MAX") ? atoi(getenv("OMK_FC0_SPLITK_MAX")) : -1;
    // the fine chunking writes three times the partial sums: its split-K path pays up to 1024 rows only (measured)
    const int splitk_max = splitk_env >= 0 ? splitk_env : (fine ? 1024 : kSplitKMaxRows);
    if (rows_bound <= splitk_max) {
        // Small and medium batches (a single game's rounds of 8, Agent::new, an arena of 100 games, ...): the pair kernel
        // would stream all of K through a handful of CTA pairs (0.18 ms however few tiles there are); instead every
        // (128-row tile, N half, chunk) is one CTA and k_fc0_reduce adds the chunks in order.
        const int kChunks = F_K0 / F_BK / (fine ? F_CHUNK0_FINE : F_CHUNK0);
        const int mt = (rows_bound + F_BM - 1) / F_BM, ws_rows = mt * F_BM;
        // per workspace: two search lanes may run this path at the same time
        if (c->ws.splitk_partial.grow(c->stream, (size_t)kChunks * ws_rows * F_N) != cudaSuccess) return false;
        float *partial = c->ws.splitk_partial;
        static const int narrow_env = getenv("OMK_FC0_SPLITK_NARROW") ? atoi(getenv("OMK_FC0_SPLITK_NARROW")) : -1;
        if (mt <= (narrow_env >= 0 ? narrow_env : 2)) {
            // one or two row tiles (a single game's rounds of 8, Agent::new): 128-column tiles double the CTAs (72 per row tile
            // instead of 36 on 148 SMs) and halve each CTA's MMA time and weight bytes.  An output element's sum does not
            // depend on the width of the tile it is computed in: same products, same chunks, same order (test_batch_invariance).
            using Cfg = FcCfg<false, 128>;
            auto sk = fine ? k_fc16<F_K0, F_CHUNK0_FINE, false, 128, false, true> : k_fc16<F_K0, F_CHUNK0, false, 128, false, true>;
            cudaFuncSetAttribute(sk, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
            sk<<<dim3(F_N / 128, mt, F_K0 / F_BK / F_SPLITK_KB), Cfg::kThreads, Cfg::kSmemBytes, c->stream>>>(
                am->map0_a_hi, am->map0_a_lo, m.map0_b_hi, m.map0_b_lo, m.t[24], m.fc_inv_scale, partial, nullptr,
                nullptr, c->ws.n_req, rows_bound, nullptr, nullptr, nullptr, FcBal{});
        } else {
            using Cfg = FcCfg<false, 256>;
            auto sk = fine ? k_fc16<F_K0, F_CHUNK0_FINE, false, 256, false, true> : k_fc16<F_K0, F_CHUNK0, false, 256, false, true>;
            cudaFuncSetAttribute(sk, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
            sk<<<dim3(F_N / F_BN, mt, F_K0 / F_BK / F_SPLITK_KB), Cfg::kThreads, Cfg::kSmemBytes, c->stream>>>(
                am->map0_a_hi, am->map0_a_lo, m.map0s_b_hi, m.map0s_b_lo, m.t[24], m.fc_inv_scale, partial, nullptr,
                nullptr, c->ws.n_req, rows_bound, nullptr, nullptr, nullptr, FcBal{});
        }
        k_fc0_reduce<<<(rows_bound * 64 + 255) / 256, 256, 0, c->stream>>>(partial, kChunks, ws_rows, m.t[24],
                                                                            m.fc_inv_scale, c->ws.act1_h16, c->ws.act1_l16,
                                                                            c->ws.n_req, rows_bound);
        c->launches += 2;
        return check_launch("fc0 (fp16 split, split-K)");
    }
    auto kern = fine ? k_fc16<F_K0, F_CHUNK0_FINE, true> : k_fc16<F_K0, F_CHUNK0, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FcCfg<true, 256>::kSmemBytes);
    const int pairs = (rows_bound + 255) / 256;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * (F_N / F_BN) * pairs, 1);
    cfg.blockDim = dim3(FcCfg<true, 256>::kThreads);
    cfg.dynamicSmemBytes = FcCfg<true, 256>::kSmemBytes;
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const float *bias_p = m.t[24];
    const float *inv_p = m.fc_inv_scale;
    float *c_f32 = nullptr;
    __half *c_hi = c->ws.act1_h16, *c_lo = c->ws.act1_l16;
    const uint32_t *nreq_p = c->ws.n_req;
    float *no_p = nullptr, *no_v = nullptr;
    uint32_t *no_err = nullptr;
    // tail balancing (see FcBal): the last, partial wave of tiles shares its K range with the otherwise idle pairs
    FcBal bal{};
    if (!fine && c->fc0_balance) {
        Fc16State *st = state16_of(c);
        if (st->pair_slots == 0) {
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
            st->pair_slots = n > 0 ? n : -1;
        }
        const int P = st->pair_slots, T = (F_N / F_BN) * pairs, NC = F_K0 / F_BK / F_CHUNK0;
        const int R = P > 0 ? T % P : 0, H = P - R;
        if (R > 0 && R <= 128 && H > 0) {
            int tail = 0;
            for (int t = 1; t <= F_BAL_TAIL_MAX; ++t)
                if ((R * t + H - 1) / H + 1 <= NC - t) tail = t;  // the helpers' units fit beside the mains' own chunks
            if (tail > 0) {
                const int units = R * tail;
                bool ok = true;
                Workspace &w = c->ws;
                if (!w.bal_flags)
                    ok = w.bal_flags.alloc(256) == cudaSuccess && cudaMemsetAsync(w.bal_flags, 0, w.bal_flags.bytes(), c->stream) == cudaSuccess;
                if (!ok || w.bal_partial.grow(c->stream, F_BAL_UNIT_F4 * (size_t)units) != cudaSuccess) return false;
                bal.full = T - R;
                bal.helpers = H;
                bal.mains = R;
                bal.tail = tail;
                bal.m = NC - tail;
                bal.partial = w.bal_partial;
                bal.flags = w.bal_flags;
                cfg.gridDim = dim3(2 * (T + H), 1);
            }
        }
    }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, am->map0_a_hi, am->map0_a_lo, m.map0_b_hi, m.map0_b_lo, bias_p, inv_p, c_f32,
                                             c_hi, c_lo, nreq_p, rows_bound, no_p, no_v, no_err, bal);
    if (e != cudaSuccess) fprintf(stderr, "omok_b200: cudaLaunchKernelEx(k_fc16 pair): %s\n", cudaGetErrorString(e));
    c->launches++;
    return e == cudaSuccess && check_launch("fc0 (fp16 split)");
}

// fc1: act1_h16/l16 -> act2_h16/l16 (the A operand of the heads)
bool launch_fc1_f16(omk_ctx *c, int rows_bound) {
    const NetWeights &m = *c->model;
    const ActMaps *am = m.weights_ready ? &c->ws.maps : nullptr;
    if (!am) return false;
    using Cfg = FcCfg<false, 256>;
    auto kern = k_fc16<F_K1, F_CHUNK1, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    const int mt = (rows_bound + F_BM - 1) / F_BM;
    kern<<<dim3(F_N / F_BN, mt), Cfg::kThreads, Cfg::kSmemBytes, c->stream>>>(
        am->map1_a_hi, am->map1_a_lo, m.map1_b_hi, m.map1_b_lo, m.t[26], m.fc_inv_scale + 1, nullptr, c->ws.act2_h16,
        c->ws.act2_l16, c->ws.n_req, rows_bound, nullptr, nullptr, nullptr, FcBal{});
    c->launches++;
    return check_launch("fc1 (fp16 split)");
}

// heads: act2_h16/l16 -> P (softmax of the 81 policy logits) and V (tanh of the value logit), or with `logits` the 82
// logits into ws.logits
bool launch_heads_f16(omk_ctx *c, int rows_bound, bool logits) {
    const NetWeights &m = *c->model;
    const ActMaps *am = m.weights_ready ? &c->ws.maps : nullptr;
    if (!am) return false;
    using Cfg = FcCfg<false, 128>;
    auto kern = logits ? k_fc16<F_K1, F_CHUNKH, false, 128, true, false, true> : k_fc16<F_K1, F_CHUNKH, false, 128, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    const int mt = (rows_bound + F_BM - 1) / F_BM;
    kern<<<dim3(1, mt), Cfg::kThreads, Cfg::kSmemBytes, c->stream>>>(
        am->map2_a_hi, am->map2_a_lo, m.map2_b_hi, m.map2_b_lo, m.heads_b, m.fc_inv_scale + 2, logits ? c->ws.logits.get() : nullptr,
        nullptr, nullptr, c->ws.n_req, rows_bound, logits ? nullptr : c->ws.P.get(), logits ? nullptr : c->ws.V.get(), c->dev_error,
        FcBal{});
    c->launches++;
    return check_launch("heads (fp16 split)");
}

}  // namespace omk
