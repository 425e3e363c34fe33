// train_kernels.cu -- the trainer's gradient step behind the C ABI (omk_train_step): AgentModel::train of the reference
// (alpha-zero/src/agent_model.rs:26-103,136-168) as plain fp32 CUDA kernels.
//
//   loss   = mean((z - v)^2) over axes [0,1]  +  mean(softmax_cross_entropy_with_logits(logits, pi)) over axis 0
//            (agent_model.rs:60-73, network.rs:249-253)
//   update = tensorflow::train::AdadeltaOptimizer, learning rate 0.01 (agent_model.rs:24,75-83), rho 0.95 and
//            epsilon 1e-8 (the crate's defaults) == the ApplyAdadelta op:
//                accum        = rho * accum + (1 - rho) * g^2
//                update       = sqrt(accum_update + eps) / sqrt(accum + eps) * g
//                var         -= lr * update
//                accum_update = rho * accum_update + (1 - rho) * update^2
//   train() = one minimize step, then a SECOND forward that reports (p_loss, v_loss, loss) (agent_model.rs:150-167).
//
// This is NOT the self-play hot path: an iteration runs 600 steps of 128 positions against ~10^8 network evaluations
// of self-play, so the kernels here are written for correctness and determinism (fp32 everywhere, fixed summation
// orders, no floating-point atomics), not for the tensor cores: one generic tiled GEMM with transposes, K slicing and
// fused epilogues (bias, residual, lrelu, the lrelu' gate of the backward pass, the bias gradient of a weight-gradient
// product), the depthwise forward / data-gradient / weight-gradient kernels, the loss, and the optimizer.  At the
// reference's own iteration shape (50 episodes, 600 updates) the step is most of an iteration on the GPU, so its
// launch count and its low-parallelism reductions were worth fixing: 3.2 -> 1.2 ms per 128 positions
// (profiles/r02_train_step.md).
// Data parallelism (BASELINE config 5): the flat gradient (5 643 250 floats, 22.6 MB) is all-reduced over NCCL when a
// communicator is attached (omk_train_comm_init; libnccl is loaded with dlopen, the library has no link dependency on
// it) or handed to the caller between omk_train_backward and omk_train_apply.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>

#include "omk_internal.h"

namespace omk {

constexpr int kTP = 128, kTM = 32, kTF = 512, kTFlat = kCells * kTP;  // channels, bottleneck width, fc width, 10368
constexpr float kTLrelu = 0.2f;  // TensorFlow LeakyRelu default alpha

static const long long kTLen[kNetTensors] = {
    384, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    (long long)kTFlat * kTF, kTF, kTF * kTF, kTF, kTF, 1, kTF * kCells, kCells};
constexpr long long kTParams = 5643250;

// ---------------------------------------------------------------------------------------------------------------
// C[M,N] = epilogue( op(A) . op(B) ), fp32, 64x64x16 tiles, 256 threads, 4x4 outputs per thread.
//   TA: A is stored [K,M] (row-major) and read transposed; TB: B is stored [N,K].
//   epilogue: (+ bias[n]) (+ res[m,n]) (lrelu if act) (+ C if accumulate) (* lrelu'(gate[m,n]) if gate)
// K is walked in order by one CTA per output tile: the summation order of an output element is fixed.
// ---------------------------------------------------------------------------------------------------------------
struct GemmEpi {
    const float *bias = nullptr;  // [N]
    const float *res = nullptr;   // [M,N], leading dimension ldc
    const float *gate = nullptr;  // [M,N], leading dimension ldc: multiply by (gate > 0 ? 1 : 0.2)
    int act = 0;                  // lrelu on the result
    int accumulate = 0;           // C += result
    float *colsum = nullptr;      // [N]: also the column sums of op(B) over K (a weight-gradient product X^T . dY carries the
                                  // bias gradient sum_rows dY with it: the CTAs of the first output row tile add up the B slices
                                  // they stage anyway; K slices are added in slice order by k_tgemm_reduce)
};

// Split-K (gridDim.z > 1, products with K in the thousands and few output tiles: the weight gradients of the 1x1
// convolutions, fc0's forward): slice z walks k in [z * k_per_split, (z + 1) * k_per_split) and stores its raw partial tile
// to part[z][M][N]; k_tgemm_reduce adds the slices IN ORDER and applies the epilogue -- still a fixed summation order.
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
    k_tgemm(const float *__restrict__ A, const float *__restrict__ B, float *__restrict__ C, int M, int N, int K, int lda, int ldb,
            int ldc, GemmEpi e, int k_per_split, float *__restrict__ part) {
    __shared__ __align__(16) float As[16][64 + 4];  // rows 16-byte aligned: the 4 x 4 register tile reads its operands as float4
    __shared__ __align__(16) float Bs[16][64 + 4];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    const int k_begin = (int)blockIdx.z * k_per_split, k_end = min(K, k_begin + k_per_split);
    const bool want_cs = e.colsum != nullptr && blockIdx.y == 0 && ty == 0;  // 16 threads x 4 columns of this n tile
    float cs[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    // The next k-step's 64 x 16 slice of op(A) and 16 x 64 slice of op(B) are fetched into registers while this one is
    // multiplied (a CTA with a long K and few neighbours is otherwise a chain of exposed global-load latencies: 2.4 us per
    // k-step measured); out-of-range elements are zeros.  The summation order is unchanged.
    float ra[4], rb[4];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = t + 256 * i;  // 0..1023
            int m, k;
            if (TA) { m = idx & 63; k = idx >> 6; } else { k = idx & 15; m = idx >> 4; }
            const int gm = m0 + m, gk = k0 + k;
            ra[i] = 0.0f;
            if (gm < M && gk < k_end) ra[i] = TA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
            int n, kb;
            if (TB) { kb = idx & 15; n = idx >> 4; } else { n = idx & 63; kb = idx >> 6; }
            const int gn = n0 + n, gkb = k0 + kb;
            rb[i] = 0.0f;
            if (gn < N && gkb < k_end) rb[i] = TB ? B[(size_t)gn * ldb + gkb] : B[(size_t)gkb * ldb + gn];
        }
    };
    if (k_begin < k_end) fetch(k_begin);
    for (int k0 = k_begin; k0 < k_end; k0 += 16) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = t + 256 * i;
            if (TA) As[idx >> 6][idx & 63] = ra[i]; else As[idx & 15][idx >> 4] = ra[i];
            if (TB) Bs[idx & 15][idx >> 4] = rb[i]; else Bs[idx >> 6][idx & 63] = rb[i];
        }
        __syncthreads();
        if (k0 + 16 < k_end) fetch(k0 + 16);
        if (want_cs) {
#pragma unroll
            for (int k = 0; k < 16; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) cs[j] += Bs[k][tx * 4 + j];
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float4 a4 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]), b4 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    if (want_cs) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            if (part) part[(size_t)gridDim.z * M * N + (size_t)blockIdx.z * N + n] = cs[j];  // slice sums behind the partial tiles
            else e.colsum[n] = cs[j];
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (part) {  // split-K slice: raw partial sums, the epilogue runs in k_tgemm_reduce
                part[((size_t)blockIdx.z * M + m) * N + n] = v;
                continue;
            }
            const size_t o = (size_t)m * ldc + n;
            if (e.bias) v += e.bias[n];
            if (e.res) v += e.res[o];
            if (e.act) v = v > 0.0f ? v : kTLrelu * v;
            if (e.accumulate) v += C[o];
            if (e.gate) v *= e.gate[o] > 0.0f ? 1.0f : kTLrelu;
            C[o] = v;
        }
    }
}

__global__ void k_tgemm_reduce(const float *__restrict__ part, int splits, int M, int N, float *__restrict__ C, int ldc, GemmEpi e) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)M * N) return;
    if (e.colsum && idx < N) {  // the K slices' column sums of op(B), in slice order
        const float *pc = part + (size_t)splits * M * N + idx;
        float cs = 0.0f;
        for (int z = 0; z < splits; ++z) cs += pc[(size_t)z * N];
        e.colsum[idx] = cs;
    }
    const int m = (int)(idx / N), n = (int)(idx % N);
    float v = 0.0f;
    int z = 0;
    for (; z + 4 <= splits; z += 4) {  // four independent loads in flight, added in slice order
        const float p0 = part[((size_t)z * M + m) * N + n], p1 = part[((size_t)(z + 1) * M + m) * N + n],
                    p2 = part[((size_t)(z + 2) * M + m) * N + n], p3 = part[((size_t)(z + 3) * M + m) * N + n];
        v += p0; v += p1; v += p2; v += p3;
    }
    for (; z < splits; ++z) v += part[((size_t)z * M + m) * N + n];
    const size_t o = (size_t)m * ldc + n;
    if (e.bias) v += e.bias[n];
    if (e.res) v += e.res[o];
    if (e.act) v = v > 0.0f ? v : kTLrelu * v;
    if (e.accumulate) v += C[o];
    if (e.gate) v *= e.gate[o] > 0.0f ? 1.0f : kTLrelu;
    C[o] = v;
}

static float *g_splitk_scratch(omk_ctx *c, size_t floats);  // grow-only scratch of the training state

template <bool TA, bool TB>
static void tgemm(omk_ctx *c, const float *A, const float *B, float *C, int M, int N, int K, int lda, int ldb, int ldc,
                  const GemmEpi &e) {
    cudaStream_t s = c->stream;
    dim3 grid((N + 63) / 64, (M + 63) / 64);
    // few output tiles: slice K so that ~2 waves of CTAs exist (fixed slice size -> fixed summation order).  One CTA walks
    // its K in steps of 16 with a CTA barrier each, so a 16-tile product with K = 512 (fc1 and the heads on a minibatch of
    // 128) was 32 dependent steps on 16 SMs: 85 us; sliced, 2 steps on 256 CTAs.
    const int tiles = (int)(grid.x * grid.y);
    if (K >= 128 && tiles < 592) {  // fewer than four CTAs per SM: aim at eight
        int splits = min(64, max(2, 1184 / tiles));
        int kps = max(32, ((K + splits - 1) / splits + 15) / 16 * 16);
        splits = (K + kps - 1) / kps;
        float *part = splits >= 2 ? g_splitk_scratch(c, (size_t)splits * M * N + (size_t)splits * N) : nullptr;
        if (part) {
            grid.z = splits;
            k_tgemm<TA, TB><<<grid, 256, 0, s>>>(A, B, C, M, N, K, lda, ldb, ldc, e, kps, part);
            const long long tot = (long long)M * N;
            k_tgemm_reduce<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(part, splits, M, N, C, ldc, e);
            c->launches++;
            return;
        }
    }
    k_tgemm<TA, TB><<<grid, 256, 0, s>>>(A, B, C, M, N, K, lda, ldb, ldc, e, K, nullptr);
}

constexpr int kRedSlicesMax = 64;

// depthwise 3x3, SAME zero padding, stride 1, no bias (network-utils lib.rs:204-216) on [n][81][32]; dw is [3][3][32]
// forward: out[p][c] = sum_tap in[p + tap][c] * dw[tap][c]
// data gradient (flip = 1): din[q][c] = sum_tap dout[q - tap][c] * dw[tap][c]
__global__ void k_dw(const float *__restrict__ in, const float *__restrict__ dw, float *__restrict__ out, int n, int flip,
                     const float *__restrict__ gate) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n * kCells * kTM;
    if (idx >= total) return;
    const int c = (int)(idx & 31);
    const int p = (int)((idx >> 5) % kCells);
    const long long b = (idx >> 5) / kCells;
    const int y = p / kSide, x = p % kSide;
    const float *src = in + b * kCells * kTM;
    float acc = 0.0f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int yy = flip ? y - (ky - 1) : y + (ky - 1), xx = flip ? x - (kx - 1) : x + (kx - 1);
            if (yy < 0 || yy >= kSide || xx < 0 || xx >= kSide) continue;
            acc = fmaf(src[(yy * kSide + xx) * kTM + c], dw[(ky * 3 + kx) * kTM + c], acc);
        }
    }
    if (gate) acc *= gate[idx] > 0.0f ? 1.0f : kTLrelu;
    out[idx] = acc;
}
// weight gradient: ddw[tap][c] = sum over positions b and pixels p of in[b][p + tap][c] * dout[b][p][c]
// grid (9 taps, slices of positions); a CTA = 32 channels x 8 position groups over its slice, groups added in order, and stores
// its slice sum; the LAST CTA of a tap to finish adds the slices in slice order -- whichever CTA that is, the order of the
// additions is the same, so the result is deterministic without a second launch (nine CTAs walking the whole minibatch were
// 250 us per call).  The `done` counters re-arm themselves.
__global__ void k_dw_wgrad(const float *__restrict__ in, const float *__restrict__ dout, float *__restrict__ ddw, int n,
                           float *__restrict__ slice_sums, uint32_t *__restrict__ done) {
    __shared__ float part[8][33];
    __shared__ bool last;
    const int tap = blockIdx.x, ky = tap / 3, kx = tap % 3;
    const int c = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int slices = (int)gridDim.y, per = (n + slices - 1) / slices;
    const int b_begin = (int)blockIdx.y * per, b_end = min(n, b_begin + per);
    float s = 0.0f;
    for (int b = b_begin + g; b < b_end; b += 8) {
        const float *ip = in + (size_t)b * kCells * kTM, *dp = dout + (size_t)b * kCells * kTM;
        for (int p = 0; p < kCells; ++p) {
            const int y = p / kSide + ky - 1, x = p % kSide + kx - 1;
            if (y < 0 || y >= kSide || x < 0 || x >= kSide) continue;
            s = fmaf(ip[(y * kSide + x) * kTM + c], dp[p * kTM + c], s);
        }
    }
    part[g][c] = s;
    __syncthreads();
    if (g == 0) {
        float tot = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) tot += part[i][c];
        if (slices == 1) ddw[tap * kTM + c] = tot; else slice_sums[((size_t)blockIdx.y * 9 + tap) * kTM + c] = tot;
    }
    if (slices == 1) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done + tap, 1u) == (uint32_t)slices - 1u;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (g == 0) {
        float tot = 0.0f;
        for (int z = 0; z < slices; ++z) tot += __ldcg(slice_sums + ((size_t)z * 9 + tap) * kTM + c);
        ddw[tap * kTM + c] = tot;
    }
    if (threadIdx.x == 0) done[tap] = 0u;
}

// the first maximum (lowest index among equal values) of a warp's (value, index) candidates
__device__ __forceinline__ int warp_first_argmax(float v, int idx) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, off);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, off);
        if (ov > v || (ov == v && oi < idx)) {
            v = ov;
            idx = oi;
        }
    }
    return idx;
}

// per position: softmax cross entropy with the visit policy, squared value error, and their logit gradients for the
// MEAN losses (1/n folded in).  row_loss[2*i] = policy term, [2*i+1] = value term.  Row i's logits are logits[i * lstride ..],
// its value logit vlogit[i * vstride] (the trainer: 81 and 1; omk_replay_score reads the evaluator's [rows][128] in place).
// top1 (may be nullptr): 1 if the first maximum of the logits (ascending cell order) is the first maximum of pi, else 0.
__global__ void k_loss(const float *__restrict__ logits, int lstride, const float *__restrict__ vlogit, int vstride,
                       const float *__restrict__ pi, const float *__restrict__ z, int n, float *__restrict__ dlogits,
                       float *__restrict__ dvlogit, float *__restrict__ row_loss, uint8_t *__restrict__ top1) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= n) return;
    const float *l = logits + (size_t)row * lstride, *t = pi + (size_t)row * kCells;
    float v[3], tv[3], mx = -INFINITY, tsum = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = lane + 32 * j;
        v[j] = c < kCells ? l[c] : -INFINITY;
        tv[j] = c < kCells ? t[c] : 0.0f;
        mx = fmaxf(mx, v[j]);
        tsum += tv[j];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        tsum += __shfl_xor_sync(0xffffffffu, tsum, off);
    }
    float ex[3], s = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        ex[j] = (lane + 32 * j) < kCells ? expf(v[j] - mx) : 0.0f;
        s += ex[j];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float lse = mx + logf(s), inv = 1.0f / s, invn = 1.0f / (float)n;
    float pl = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = lane + 32 * j;
        if (c < kCells) {
            pl -= tv[j] * (v[j] - lse);
            if (dlogits) dlogits[(size_t)row * kCells + c] = (ex[j] * inv * tsum - tv[j]) * invn;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) pl += __shfl_xor_sync(0xffffffffu, pl, off);
    bool agree = false;
    if (top1) {  // each lane's candidates are in ascending cell order, so a strict > keeps the first maximum
        float bl = v[0], bt = tv[0];
        int il = lane, it = lane;
#pragma unroll
        for (int j = 1; j < 3; ++j) {
            const int c = lane + 32 * j;
            if (c < kCells && v[j] > bl) { bl = v[j]; il = c; }
            if (c < kCells && tv[j] > bt) { bt = tv[j]; it = c; }
        }
        agree = warp_first_argmax(bl, il) == warp_first_argmax(bt, it);
    }
    if (lane == 0) {
        // tanh and its derivative from one exponential: 1 - tanh^2 = 4e / (1 + e)^2 with e = exp(-2|x|) keeps its relative
        // accuracy where tanh saturates (value logits have a scale of ~20; 1 - v*v would cancel to a few bits there)
        const float xl = vlogit[(size_t)row * vstride], ex2 = expf(-2.0f * fabsf(xl)), den = 1.0f + ex2;
        const float val = copysignf((1.0f - ex2) / den, xl), sech2 = 4.0f * ex2 / (den * den);
        const float d = val - z[row];
        row_loss[2 * row] = pl;
        row_loss[2 * row + 1] = d * d;
        if (dvlogit) dvlogit[row] = 2.0f * d * sech2 * invn;
        if (top1) top1[row] = agree ? 1 : 0;
    }
}
// (p_loss, v_loss, loss) = means over the rows, summed in row order by one thread per term (n is a minibatch)
__global__ void k_loss_reduce(const float *__restrict__ row_loss, int n, float *__restrict__ out3) {
    if (threadIdx.x < 2) {
        float s = 0.0f;
        for (int i = 0; i < n; ++i) s += row_loss[2 * i + threadIdx.x];
        out3[threadIdx.x] = s / (float)n;
    }
    __syncthreads();
    if (threadIdx.x == 0) out3[2] = out3[0] + out3[1];
}

// omk_replay_score's means (DESIGN.md 2): block b's three sums over rows [1024 b, 1024 b + 1024), each in row order in fp64 from
// 0.0 by one thread, so they depend on nothing but the rows; row_loss is de-interleaved into p_out / v_out on the way
constexpr int kScoreBlock = 1024;
__global__ void __launch_bounds__(kScoreBlock) k_score_reduce(const float *__restrict__ row_loss, const uint8_t *__restrict__ top1,
                                                              long long n, float *__restrict__ p_out, float *__restrict__ v_out,
                                                              double *__restrict__ block_sums) {
    __shared__ float sp[kScoreBlock], sv[kScoreBlock];
    __shared__ uint8_t st[kScoreBlock];
    const long long r0 = (long long)blockIdx.x * kScoreBlock, i = r0 + threadIdx.x;
    const int m = (int)min((long long)kScoreBlock, n - r0);
    if (threadIdx.x < m) {
        const float2 pv = reinterpret_cast<const float2 *>(row_loss)[i];
        sp[threadIdx.x] = pv.x;
        sv[threadIdx.x] = pv.y;
        st[threadIdx.x] = top1[i];
        p_out[i] = pv.x;
        v_out[i] = pv.y;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        if (threadIdx.x == 0) for (int k = 0; k < m; ++k) s += (double)sp[k];
        else if (threadIdx.x == 1) for (int k = 0; k < m; ++k) s += (double)sv[k];
        else for (int k = 0; k < m; ++k) s += (double)st[k];
        block_sums[3 * (size_t)blockIdx.x + threadIdx.x] = s;
    }
}
// the block sums in ascending block order -> {mean p_loss, mean v_loss, mean p_loss + mean v_loss, mean top1}
__global__ void k_score_means(const double *__restrict__ block_sums, int blocks, long long n, double *__restrict__ means4) {
    __shared__ double mean[3];
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int b = 0; b < blocks; ++b) s += block_sums[3 * (size_t)b + threadIdx.x];
        mean[threadIdx.x] = s / (double)n;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        means4[0] = mean[0];
        means4[1] = mean[1];
        means4[2] = mean[0] + mean[1];
        means4[3] = mean[2];
    }
}

__global__ void k_scale(float *x, long long n, float f) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] *= f;
}

// tensorflow ApplyAdadelta (see the header of this file) on all 31 tensors in one launch: the variables are separate
// allocations, the gradient and the two slot arrays are flat in checkpoint order (element i of the flat index belongs to
// the tensor whose [off[k], off[k + 1]) holds it)
struct AdadeltaTensors {
    float *var[kNetTensors];
    long long off[kNetTensors + 1];
};
__global__ void k_adadelta(const AdadeltaTensors T, float *__restrict__ accum, float *__restrict__ accum_update, const float *__restrict__ g,
                           float lr, float rho, float eps) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T.off[kNetTensors]) return;
    int k = 0;
#pragma unroll 1
    while (i >= T.off[k + 1]) ++k;
    float *var = T.var[k] + (i - T.off[k]);
    const float gi = g[i];
    const float a = rho * accum[i] + (1.0f - rho) * gi * gi;
    const float upd = sqrtf(accum_update[i] + eps) * (1.0f / sqrtf(a + eps)) * gi;
    accum[i] = a;
    *var -= lr * upd;
    accum_update[i] = rho * accum_update[i] + (1.0f - rho) * upd * upd;
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// The two buffer groups of the training state, each allocated into a local instance and committed whole (train_ensure)
struct TrainBatch {  // per-minibatch buffers, sized for cap_n positions
    int cap_n = 0;
    Buf<float> img, pi, z;
    Buf<float> x[4];                     // residual stream after the stem and after each block: [n*81][128]
    Buf<float> h0[3], hd[3], h1[3];      // per block: conv0 out, depthwise out, pointwise out: [n*81][32]
    Buf<float> a0, a1;                   // fc0 / fc1 outputs [n][512]
    Buf<float> logits, vlogit;
    Buf<float> dx, dy;                   // [n*81][128] gradient of the residual stream / of a block's pre-activation sum
    Buf<float> d32a, d32b;               // [n*81][32]
    Buf<float> da0, da1, dlogits, dvlogit, row_loss;
};
struct TrainOptimizer {
    Buf<float> grads;                    // flat [kTParams] in checkpoint order
    Buf<float> accum, accum_update;      // Adadelta slots, flat
    Buf<float> losses;                   // [3] device
    Buf<float> red_sums;                 // [kRedSlicesMax][9][32] slice sums of the depthwise weight gradients
    Buf<uint32_t> red_done;              // [32] arrival counters of that reduction (self re-arming)
};
struct TrainState : TrainBatch, TrainOptimizer {
    Buf<float> splitk;                   // split-K partial tiles (grow-only)
    long long off[kNetTensors + 1] = {};
    long long steps = 0;
    // NCCL (optional, loaded with dlopen)
    void *nccl_lib = nullptr, *comm = nullptr;
    int world = 1, rank = 0;
    int (*p_allreduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*p_comm_init_rank)(void **, int, const void * /* ncclUniqueId by value: 128 bytes */, int) = nullptr;
    int (*p_comm_destroy)(void *) = nullptr;
    const char *(*p_err)(int) = nullptr;
    ~TrainState() {
        if (comm && p_comm_destroy) p_comm_destroy(comm);
        if (nccl_lib) dlclose(nccl_lib);
    }
};
void TrainStateFree::operator()(TrainState *t) const { delete t; }
struct NcclUniqueId { char internal[128]; };

static TrainState *train_state(omk_ctx *c) {
    if (!c->train_state) {
        TrainState *t = new TrainState();
        long long o = 0;
        for (int i = 0; i < kNetTensors; ++i) {
            t->off[i] = o;
            o += kTLen[i];
        }
        t->off[kNetTensors] = o;
        c->train_state.reset(t);
    }
    return c->train_state.get();
}

static float *g_splitk_scratch(omk_ctx *c, size_t floats) {
    TrainState *t = train_state(c);
    return t->splitk.grow(c->stream, floats) == cudaSuccess ? t->splitk.get() : nullptr;
}

static bool train_ensure(omk_ctx *c, TrainState *t, int n) {
    auto ok = [](auto &b, size_t count) { return b.alloc(count) == cudaSuccess; };
    if (!t->grads) {
        TrainOptimizer o;
        if (!ok(o.grads, kTParams) || !ok(o.accum, kTParams) || !ok(o.accum_update, kTParams) || !ok(o.losses, 4) ||
            !ok(o.red_sums, (size_t)kRedSlicesMax * kTF) || !ok(o.red_done, 32))
            return false;
        cudaMemsetAsync(o.accum, 0, o.accum.bytes(), c->stream);
        cudaMemsetAsync(o.accum_update, 0, o.accum_update.bytes(), c->stream);
        cudaMemsetAsync(o.red_done, 0, o.red_done.bytes(), c->stream);
        static_cast<TrainOptimizer &>(*t) = std::move(o);
    }
    if (n <= t->cap_n) return true;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return false;
    static_cast<TrainBatch &>(*t) = TrainBatch{};  // the old buffers go before the new ones are allocated
    const size_t N = (size_t)n, M = N * kCells;
    TrainBatch b;
    bool all = ok(b.img, N * 243) && ok(b.pi, N * kCells) && ok(b.z, N);
    for (int i = 0; i < 4; ++i) all = all && ok(b.x[i], M * kTP);
    for (int r = 0; r < 3; ++r) all = all && ok(b.h0[r], M * kTM) && ok(b.hd[r], M * kTM) && ok(b.h1[r], M * kTM);
    all = all && ok(b.a0, N * kTF) && ok(b.a1, N * kTF) && ok(b.logits, N * kCells) && ok(b.vlogit, N) && ok(b.dx, M * kTP) &&
          ok(b.dy, M * kTP) && ok(b.d32a, M * kTM) && ok(b.d32b, M * kTM) && ok(b.da0, N * kTF) && ok(b.da1, N * kTF) &&
          ok(b.dlogits, N * kCells) && ok(b.dvlogit, N) && ok(b.row_loss, 2 * N);
    if (!all) return false;
    b.cap_n = n;
    static_cast<TrainBatch &>(*t) = std::move(b);
    return true;
}

// tensor indices in checkpoint order
enum { T_CONV_W = 0, T_CONV_B = 1, T_BLK0 = 2, T_FC0_W = 23, T_FC0_B = 24, T_FC1_W = 25, T_FC1_B = 26, T_V_W = 27, T_V_B = 28, T_P_W = 29, T_P_B = 30 };
enum { B_W0 = 0, B_B0 = 1, B_DW = 2, B_PW = 3, B_B1 = 4, B_W2 = 5, B_B2 = 6 };

// the reference network in fp32, keeping every layer the backward pass needs (network.rs:51-262)
static void train_forward(omk_ctx *c, TrainState *t, int n) {
    cudaStream_t s = c->stream;
    const Buf<float> *W = c->net.t;
    const int M = n * kCells;
    GemmEpi e;
    e.bias = W[T_CONV_B];
    e.act = 1;
    tgemm<false, false>(c, t->img, W[T_CONV_W], t->x[0], M, kTP, 3, 3, kTP, kTP, e);  // stem: the 243-float slot read as [81][3]
    for (int r = 0; r < 3; ++r) {
        const Buf<float> *B = W + T_BLK0 + 7 * r;
        GemmEpi e0;
        e0.bias = B[B_B0];
        e0.act = 1;
        tgemm<false, false>(c, t->x[r], B[B_W0], t->h0[r], M, kTM, kTP, kTP, kTM, kTM, e0);
        const long long tot = (long long)M * kTM;
        k_dw<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(t->h0[r], B[B_DW], t->hd[r], n, 0, nullptr);
        GemmEpi e1;
        e1.bias = B[B_B1];
        e1.act = 1;
        tgemm<false, false>(c, t->hd[r], B[B_PW], t->h1[r], M, kTM, kTM, kTM, kTM, kTM, e1);
        GemmEpi e2;
        e2.bias = B[B_B2];
        e2.res = t->x[r];
        e2.act = 1;
        tgemm<false, false>(c, t->h1[r], B[B_W2], t->x[r + 1], M, kTP, kTM, kTM, kTP, kTP, e2);
    }
    GemmEpi f0;
    f0.bias = W[T_FC0_B];
    f0.act = 1;
    tgemm<false, false>(c, t->x[3], W[T_FC0_W], t->a0, n, kTF, kTFlat, kTFlat, kTF, kTF, f0);  // NHWC flatten == the row itself
    GemmEpi f1;
    f1.bias = W[T_FC1_B];
    f1.act = 1;
    tgemm<false, false>(c, t->a0, W[T_FC1_W], t->a1, n, kTF, kTF, kTF, kTF, kTF, f1);
    GemmEpi hp;
    hp.bias = W[T_P_B];
    tgemm<false, false>(c, t->a1, W[T_P_W], t->logits, n, kCells, kTF, kTF, kCells, kCells, hp);
    GemmEpi hv;
    hv.bias = W[T_V_B];
    tgemm<false, false>(c, t->a1, W[T_V_W], t->vlogit, n, 1, kTF, kTF, 1, 1, hv);
    c->launches += 5 + 3 * 4;
}

static void train_losses(omk_ctx *c, TrainState *t, int n, bool with_grads) {
    k_loss<<<(n + 7) / 8, 256, 0, c->stream>>>(t->logits, kCells, t->vlogit, 1, t->pi, t->z, n, with_grads ? t->dlogits.get() : nullptr,
                                                with_grads ? t->dvlogit.get() : nullptr, t->row_loss, nullptr);
    k_loss_reduce<<<1, 32, 0, c->stream>>>(t->row_loss, n, t->losses);
    c->launches += 2;
}

// gradients of the mean loss with respect to all 31 tensors, into t->grads (checkpoint order)
static void train_backward(omk_ctx *c, TrainState *t, int n) {
    cudaStream_t s = c->stream;
    const Buf<float> *W = c->net.t;
    const int M = n * kCells;
    auto G = [&](int tensor) { return t->grads + t->off[tensor]; };
    GemmEpi none;
    auto with_colsum = [](float *bias_grad) { GemmEpi e; e.colsum = bias_grad; return e; };  // weight gradient + its bias gradient
    // heads
    tgemm<true, false>(c, t->a1, t->dlogits, G(T_P_W), kTF, kCells, n, kTF, kCells, kCells, with_colsum(G(T_P_B)));   // a1^T . dlogits
    tgemm<true, false>(c, t->a1, t->dvlogit, G(T_V_W), kTF, 1, n, kTF, 1, 1, with_colsum(G(T_V_B)));
    tgemm<false, true>(c, t->dlogits, W[T_P_W], t->da1, n, kTF, kCells, kCells, kCells, kTF, none);  // dlogits . Pw^T
    {   // da1 = (dlogits . Pw^T + dvlogit . Vw^T) * lrelu'(a1): the second product accumulates and applies the gate
        GemmEpi e;
        e.accumulate = 1;
        e.gate = t->a1;
        tgemm<false, true>(c, t->dvlogit, W[T_V_W], t->da1, n, kTF, 1, 1, 1, kTF, e);
    }
    // fc1
    tgemm<true, false>(c, t->a0, t->da1, G(T_FC1_W), kTF, kTF, n, kTF, kTF, kTF, with_colsum(G(T_FC1_B)));
    GemmEpi g0;
    g0.gate = t->a0;
    tgemm<false, true>(c, t->da1, W[T_FC1_W], t->da0, n, kTF, kTF, kTF, kTF, kTF, g0);
    // fc0
    tgemm<true, false>(c, t->x[3], t->da0, G(T_FC0_W), kTFlat, kTF, n, kTFlat, kTF, kTF, with_colsum(G(T_FC0_B)));
    // d(flat) == d(x3) as [M][128]; every gradient of the residual stream is needed only THROUGH the lrelu that produced the
    // stream (network.rs:108-111), so the producing GEMM applies that gate in its epilogue instead of a separate pass
    float *dy = t->dy, *dx = t->dx;
    GemmEpi gx3;
    gx3.gate = t->x[3];
    tgemm<false, true>(c, t->da0, W[T_FC0_W], dy, n, kTFlat, kTF, kTF, kTF, kTFlat, gx3);
    c->launches += 9;
    // residual blocks, last to first (network-utils lib.rs:386-461; network.rs:108-111)
    for (int r = 2; r >= 0; --r) {
        const Buf<float> *B = W + T_BLK0 + 7 * r;
        const int gb = T_BLK0 + 7 * r;
        const long long tot32 = (long long)M * kTM;
        // (dy = the gradient through the block's last lrelu, written by the GEMM before this block)
        tgemm<true, false>(c, t->h1[r], dy, G(gb + B_W2), kTM, kTP, M, kTM, kTP, kTP, with_colsum(G(gb + B_B2)));
        GemmEpi g1;
        g1.gate = t->h1[r];
        tgemm<false, true>(c, dy, B[B_W2], t->d32a, M, kTM, kTP, kTP, kTP, kTM, g1);  // d(pointwise pre-activation)
        tgemm<true, false>(c, t->hd[r], t->d32a, G(gb + B_PW), kTM, kTM, M, kTM, kTM, kTM, with_colsum(G(gb + B_B1)));
        tgemm<false, true>(c, t->d32a, B[B_PW], t->d32b, M, kTM, kTM, kTM, kTM, kTM, none);  // d(depthwise output)
        k_dw_wgrad<<<dim3(9, min(kRedSlicesMax, max(1, n / 8))), 256, 0, s>>>(t->h0[r], t->d32b, G(gb + B_DW), n, t->red_sums, t->red_done);
        k_dw<<<(unsigned)((tot32 + 255) / 256), 256, 0, s>>>(t->d32b, B[B_DW], t->d32a, n, 1, t->h0[r]);  // d(conv0 pre-activation)
        tgemm<true, false>(c, t->x[r], t->d32a, G(gb + B_W0), kTP, kTM, M, kTP, kTM, kTM, with_colsum(G(gb + B_B0)));
        GemmEpi skip;  // (dy (the skip connection) + d(conv0 pre-activation) . W0^T) * lrelu'(x_r): the next block's (or the stem's) dy
        skip.res = dy;
        skip.gate = t->x[r];
        tgemm<false, true>(c, t->d32a, B[B_W0], dx, M, kTP, kTM, kTM, kTM, kTP, skip);
        float *tmp = dy; dy = dx; dx = tmp;
        c->launches += 8;
    }
    // stem
    tgemm<true, false>(c, t->img, dy, G(T_CONV_W), 3, kTP, M, 3, kTP, kTP, with_colsum(G(T_CONV_B)));
    c->launches += 1;
}

static bool train_upload(omk_ctx *c, TrainState *t, const float *images, const float *pi, const float *z, int n) {
    c->h2d_bytes += (int64_t)sizeof(float) * (int64_t)n * (243 + kCells + 1);
    return cudaMemcpyAsync(t->img, images, sizeof(float) * (size_t)n * 243, cudaMemcpyHostToDevice, c->stream) == cudaSuccess &&
           cudaMemcpyAsync(t->pi, pi, sizeof(float) * (size_t)n * kCells, cudaMemcpyHostToDevice, c->stream) == cudaSuccess &&
           cudaMemcpyAsync(t->z, z, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
}

// ---- entry points used by omk_api.cu ----
// forward + losses + backward on the local minibatch: the flat gradient of the MEAN loss is left in the gradient buffer
const char *train_backward_step(omk_ctx *c, const float *images, const float *pi, const float *z, int n, float **grads_dev) {
    TrainState *t = train_state(c);
    if (!train_ensure(c, t, n)) return "training workspace allocation failed";
    if (!train_upload(c, t, images, pi, z, n)) return "copying the minibatch to the device failed";
    if (grads_dev) *grads_dev = t->grads;
    return train_backward_resident(c, n);
}

// the replay path writes the minibatch into these buffers on the device instead of train_upload's copies
const char *train_minibatch_buffers(omk_ctx *c, int n, float **img, float **pi, float **z) {
    TrainState *t = train_state(c);
    if (!train_ensure(c, t, n)) return "training workspace allocation failed";
    *img = t->img;
    *pi = t->pi;
    *z = t->z;
    return nullptr;
}

// forward + losses + backward on the minibatch already in the workspace
const char *train_backward_resident(omk_ctx *c, int n) {
    TrainState *t = train_state(c);
    train_forward(c, t, n);
    train_losses(c, t, n, true);
    train_backward(c, t, n);
    return cudaPeekAtLastError() == cudaSuccess ? nullptr : cudaGetErrorString(cudaGetLastError());
}

// all-reduce (when a communicator is attached) + Adadelta on every tensor.  The caller re-packs the tensor-core weights.
const char *train_apply_step(omk_ctx *c) {
    TrainState *t = train_state(c);
    if (!t->grads) return "omk_train_backward has not run";
    if (t->comm && t->world > 1) {
        const int rc = t->p_allreduce(t->grads, t->grads, (size_t)kTParams, 7 /* ncclFloat32 */, 0 /* ncclSum */, t->comm, c->stream);
        if (rc != 0) return t->p_err ? t->p_err(rc) : "ncclAllReduce failed";
        k_scale<<<(unsigned)((kTParams + 255) / 256), 256, 0, c->stream>>>(t->grads, kTParams, 1.0f / (float)t->world);
        c->launches++;
    }
    AdadeltaTensors T;
    for (int i = 0; i < kNetTensors; ++i) T.var[i] = c->net.t[i];
    for (int i = 0; i <= kNetTensors; ++i) T.off[i] = t->off[i];
    k_adadelta<<<(unsigned)((kTParams + 255) / 256), 256, 0, c->stream>>>(T, t->accum, t->accum_update, t->grads, 0.01f, 0.95f, 1e-8f);
    c->launches++;
    t->steps++;
    return cudaPeekAtLastError() == cudaSuccess ? nullptr : cudaGetErrorString(cudaGetLastError());
}

// the reference's second forward: (p_loss, v_loss, loss) of the minibatch uploaded by train_backward_step, with the
// CURRENT weights; averaged over the ranks when a communicator is attached
static const char *report_forward(omk_ctx *c, TrainState *t, int n) {
    if (n > t->cap_n || n <= 0) return "no minibatch on the device";
    train_forward(c, t, n);
    train_losses(c, t, n, false);
    if (t->comm && t->world > 1) {
        const int rc = t->p_allreduce(t->losses, t->losses, 3, 7, 0, t->comm, c->stream);
        if (rc != 0) return t->p_err ? t->p_err(rc) : "ncclAllReduce failed";
        k_scale<<<1, 32, 0, c->stream>>>(t->losses, 3, 1.0f / (float)t->world);
        c->launches++;
    }
    return nullptr;
}
const char *train_report_losses_device(omk_ctx *c, int n, float *dst3) {
    TrainState *t = train_state(c);
    if (const char *e = report_forward(c, t, n)) return e;
    if (cudaMemcpyAsync(dst3, t->losses, sizeof(float) * 3, cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess) return "loss copy failed";
    return cudaPeekAtLastError() == cudaSuccess ? nullptr : cudaGetErrorString(cudaGetLastError());
}
const char *train_report_losses(omk_ctx *c, int n, float *out3) {
    TrainState *t = train_state(c);
    if (const char *e = report_forward(c, t, n)) return e;
    c->d2h_bytes += (int64_t)sizeof(float) * 3;
    if (cudaMemcpyAsync(out3, t->losses, sizeof(float) * 3, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return "loss copy failed";
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return "stream synchronisation failed";
    return cudaPeekAtLastError() == cudaSuccess ? nullptr : cudaGetErrorString(cudaGetLastError());
}

void launch_loss_rows(omk_ctx *c, const float *logits, int lstride, const float *vlogit, int vstride, const float *pi, const float *z,
                      int n, float *row_loss, uint8_t *top1) {
    k_loss<<<(n + 7) / 8, 256, 0, c->stream>>>(logits, lstride, vlogit, vstride, pi, z, n, nullptr, nullptr, row_loss, top1);
    c->launches++;
}
void launch_score_reduce(omk_ctx *c, const float *row_loss, const uint8_t *top1, long long n, float *p_out, float *v_out,
                         double *block_sums, double *means4) {
    const int blocks = (int)((n + kScoreBlock - 1) / kScoreBlock);
    k_score_reduce<<<blocks, kScoreBlock, 0, c->stream>>>(row_loss, top1, n, p_out, v_out, block_sums);
    k_score_means<<<1, 32, 0, c->stream>>>(block_sums, blocks, n, means4);
    c->launches += 2;
}

float *train_grad_buffer(omk_ctx *c) { return train_state(c)->grads; }
long long train_steps(omk_ctx *c) { return c->train_state ? train_state(c)->steps : 0; }
void train_reset_optimizer(omk_ctx *c) {
    TrainState *t = train_state(c);
    if (t->accum) {
        cudaMemsetAsync(t->accum, 0, sizeof(float) * kTParams, c->stream);
        cudaMemsetAsync(t->accum_update, 0, sizeof(float) * kTParams, c->stream);
    }
    t->steps = 0;
}
const char *train_optimizer_slots(omk_ctx *c, bool create, float **accum, float **accum_update) {
    *accum = *accum_update = nullptr;
    if (!c->train_state && !create) return nullptr;
    TrainState *t = train_state(c);
    if (!t->grads && create) {
        if (!train_ensure(c, t, 0)) return "optimizer state allocation failed";
        // no gradient yet: omk_train_get_grads reads zeros rather than uninitialised memory
        if (cudaMemsetAsync(t->grads, 0, t->grads.bytes(), c->stream) != cudaSuccess) return "optimizer state initialisation failed";
    }
    *accum = t->accum;
    *accum_update = t->accum_update;
    return nullptr;
}

// ---- NCCL through dlopen ----
static const char *nccl_load(TrainState *t) {
    if (t->nccl_lib) return nullptr;
    const char *names[] = {getenv("OMK_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
        if (!nm || !*nm) continue;
        t->nccl_lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (t->nccl_lib) break;
    }
    if (!t->nccl_lib) return "libnccl.so.2 not found (set OMK_NCCL_LIB to its path)";
    t->p_allreduce = reinterpret_cast<decltype(t->p_allreduce)>(dlsym(t->nccl_lib, "ncclAllReduce"));
    t->p_comm_destroy = reinterpret_cast<decltype(t->p_comm_destroy)>(dlsym(t->nccl_lib, "ncclCommDestroy"));
    t->p_err = reinterpret_cast<decltype(t->p_err)>(dlsym(t->nccl_lib, "ncclGetErrorString"));
    if (!t->p_allreduce || !dlsym(t->nccl_lib, "ncclCommInitRank") || !dlsym(t->nccl_lib, "ncclGetUniqueId")) return "libnccl lacks the expected symbols";
    return nullptr;
}
const char *train_comm_unique_id(omk_ctx *c, uint8_t *out128) {
    TrainState *t = train_state(c);
    if (const char *e = nccl_load(t)) return e;
    auto fn = reinterpret_cast<int (*)(NcclUniqueId *)>(dlsym(t->nccl_lib, "ncclGetUniqueId"));
    NcclUniqueId id;
    const int rc = fn(&id);
    if (rc != 0) return t->p_err ? t->p_err(rc) : "ncclGetUniqueId failed";
    memcpy(out128, id.internal, 128);
    return nullptr;
}
const char *train_comm_init(omk_ctx *c, const uint8_t *id128, int nranks, int rank) {
    TrainState *t = train_state(c);
    if (const char *e = nccl_load(t)) return e;
    if (t->comm && t->p_comm_destroy) {
        t->p_comm_destroy(t->comm);
        t->comm = nullptr;
    }
    auto fn = reinterpret_cast<int (*)(void **, int, NcclUniqueId, int)>(dlsym(t->nccl_lib, "ncclCommInitRank"));
    NcclUniqueId id;
    memcpy(id.internal, id128, 128);
    const int rc = fn(&t->comm, nranks, id, rank);
    if (rc != 0) return t->p_err ? t->p_err(rc) : "ncclCommInitRank failed";
    t->world = nranks;
    t->rank = rank;
    return nullptr;
}
const char *train_comm_destroy(omk_ctx *c) {
    TrainState *t = train_state(c);
    if (t->comm && t->p_comm_destroy) t->p_comm_destroy(t->comm);
    t->comm = nullptr;
    t->world = 1;
    t->rank = 0;
    return nullptr;
}

}  // namespace omk
