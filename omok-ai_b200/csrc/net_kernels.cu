// net_kernels.cu -- K3: network forward orchestration (net_forward) and the fp32 CUDA-core A/B kernels.
//
// Replaces AgentModel::{evaluate_p, evaluate_pv} (alpha-zero/src/agent_model.rs:105-134) for the
// graph built by Network::new (alpha-zero/src/network.rs:51-262) from the layer builders of
// network-utils/src/lib.rs (:95-170 conv2d+bias, :172-262 depthwise+pointwise+bias, :285-330 fc,
// :386-461 bottleneck residual).  TensorFlow's LeakyRelu default alpha 0.2 applies everywhere.
//
// Precision: the reference's random-init recipe (2/sqrt(fan_in)) produces logits with a
// standard deviation of ~22, so the north-star tolerance (1e-3 relative on priors/values) needs
// fp32-class products: one-pass TF32 misses it by 50x and bf16 by 350x (DESIGN.md 3, "Precision").
// The product path is the tcgen05 kernels of tower_f16.cu / fc_f16.cu (3-pass fp16 hi/lo split); the kernels
// in this file are the first version's fp32 CUDA-core path, kept only as an in-library A/B check of each layer
// (omk_debug_set_tower_mode / _fc0_mode = 0).  net_forward() at the bottom sequences either set.
//
// Kernels
//   k_tower : one CTA walks positions; stem 1x1 (3->128), 3x bottleneck {1x1 128->32, depthwise
//             3x3, pointwise 32->32, 1x1 32->128, +x}, everything in shared memory (all tower
//             weights resident: 116 KB), output = fc0 input row [81*128] (NHWC flatten).
//   k_gemm  : C = act(A.W + b), 128x128x16 tiles, 8x8 register tiles (fc0, fc1, heads).
//   k_heads : tanh(value logit), softmax(81 policy logits).
#include <cstdio>

#include "omk_internal.h"

namespace omk {

constexpr int kCh = 128, kMid = 32, kFc = 512, kFlat = kCells * kCh;  // 10368
constexpr float kLrelu = 0.2f;

__device__ __forceinline__ float lrelu(float v) { return v > 0.0f ? v : kLrelu * v; }

// ---- shared-memory map of k_tower (float offsets) ----
constexpr int kBlkFloats = 4096 + 32 + 288 + 1024 + 32 + 4096 + 128;  // 9696
constexpr int S_WSTEM = 0, S_BSTEM = 384, S_BLK0 = 512;
constexpr int B_W0 = 0, B_B0 = 4096, B_DW = 4128, B_PW = 4416, B_B1 = 5440, B_W2 = 5472, B_B2 = 9568;
constexpr int kXStride = 132, kHStride = 36;
constexpr int S_X = S_BLK0 + 3 * kBlkFloats;       // 29600
constexpr int S_H0 = S_X + kCells * kXStride;      // 40292
constexpr int S_H1 = S_H0 + kCells * kHStride;     // 43208
constexpr int S_IMG = S_H1 + kCells * kHStride;    // 46124
constexpr int kTowerSmemFloats = S_IMG + 256;      // 46380
constexpr int kTowerSmemBytes = kTowerSmemFloats * 4;
constexpr int kTowerThreads = 256;

struct TowerWeights {
    const float *conv_w, *conv_b;
    const float *w0[3], *b0[3], *dw[3], *pw[3], *b1[3], *w2[3], *b2[3];
};

__device__ __forceinline__ void copy_to_smem(float *dst, const float *src, int n, int t) {
    for (int i = t * 4; i < n; i += kTowerThreads * 4) *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(src + i);
}

// [81 x K] (stride SA) times [K x 32] -> [81 x 32] (stride 36), + bias, lrelu.  256 threads:
// tx = 4 output columns, ty = rows ty, ty+32, ty+64.
template <int K, int SA>
__device__ __forceinline__ void gemm_n32(const float *A, const float *W, const float *bias, float *out, int t) {
    const int tx = t & 7, ty = t >> 3;
    float acc[3][4];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    int rows[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) rows[i] = min(ty + 32 * i, kCells - 1);
#pragma unroll 4
    for (int k = 0; k < K; k += 4) {
        float4 w[4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) w[kk] = *reinterpret_cast<const float4 *>(W + (k + kk) * kMid + tx * 4);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float4 a = *reinterpret_cast<const float4 *>(A + rows[i] * SA + k);
            const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                acc[i][0] = fmaf(av[kk], w[kk].x, acc[i][0]);
                acc[i][1] = fmaf(av[kk], w[kk].y, acc[i][1]);
                acc[i][2] = fmaf(av[kk], w[kk].z, acc[i][2]);
                acc[i][3] = fmaf(av[kk], w[kk].w, acc[i][3]);
            }
        }
    }
    const float4 b = *reinterpret_cast<const float4 *>(bias + tx * 4);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int row = ty + 32 * i;
        if (row < kCells) {
            float4 o;
            o.x = lrelu(acc[i][0] + b.x);
            o.y = lrelu(acc[i][1] + b.y);
            o.z = lrelu(acc[i][2] + b.z);
            o.w = lrelu(acc[i][3] + b.w);
            *reinterpret_cast<float4 *>(out + row * kHStride + tx * 4) = o;
        }
    }
}

__global__ void __launch_bounds__(kTowerThreads, 1)
    k_tower(TowerWeights tw, const NNIn *nn_in, const float *images, const uint32_t *n_req, int max_rows, float *act0) {
    extern __shared__ __align__(16) float sm[];
    const int t = threadIdx.x;
    const int rows = (int)min(*n_req, (uint32_t)max_rows);
    if ((int)blockIdx.x >= rows) return;

    copy_to_smem(sm + S_WSTEM, tw.conv_w, 384, t);
    copy_to_smem(sm + S_BSTEM, tw.conv_b, 128, t);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        float *blk = sm + S_BLK0 + r * kBlkFloats;
        copy_to_smem(blk + B_W0, tw.w0[r], 4096, t);
        copy_to_smem(blk + B_B0, tw.b0[r], 32, t);
        copy_to_smem(blk + B_DW, tw.dw[r], 288, t);
        copy_to_smem(blk + B_PW, tw.pw[r], 1024, t);
        copy_to_smem(blk + B_B1, tw.b1[r], 32, t);
        copy_to_smem(blk + B_W2, tw.w2[r], 4096, t);
        copy_to_smem(blk + B_B2, tw.b2[r], 128, t);
    }
    float *X = sm + S_X, *H0 = sm + S_H0, *H1 = sm + S_H1, *IMG = sm + S_IMG;

    for (int row = blockIdx.x; row < rows; row += gridDim.x) {
        // ---- input image: the reference's 243-float slot, read as [81 pixels][3 channels] ----
        if (t < 243) {
            if (images) {
                IMG[t] = images[(size_t)row * 243 + t];
            } else {
                const NNIn in = nn_in[row];
                IMG[t] = image_value(in.black, in.white, in.meta & 1u, (in.meta >> 1) & 1u, t);
            }
        }
        __syncthreads();
        // ---- stem: 1x1 conv 3 -> 128, bias, lrelu (network.rs:65-79) ----
        for (int idx = t; idx < kCells * 32; idx += kTowerThreads) {
            const int pix = idx >> 5, c4 = (idx & 31) * 4;
            float4 acc = *reinterpret_cast<const float4 *>(sm + S_BSTEM + c4);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float v = IMG[3 * pix + k];
                const float4 w = *reinterpret_cast<const float4 *>(sm + S_WSTEM + k * kCh + c4);
                acc.x = fmaf(v, w.x, acc.x);
                acc.y = fmaf(v, w.y, acc.y);
                acc.z = fmaf(v, w.z, acc.z);
                acc.w = fmaf(v, w.w, acc.w);
            }
            acc.x = lrelu(acc.x); acc.y = lrelu(acc.y); acc.z = lrelu(acc.z); acc.w = lrelu(acc.w);
            *reinterpret_cast<float4 *>(X + pix * kXStride + c4) = acc;
        }
        __syncthreads();

        for (int r = 0; r < 3; ++r) {  // network-utils lib.rs:386-461
            const float *blk = sm + S_BLK0 + r * kBlkFloats;
            // conv0: 1x1 128 -> 32, bias, lrelu
            gemm_n32<kCh, kXStride>(X, blk + B_W0, blk + B_B0, H0, t);
            __syncthreads();
            // conv1 depthwise 3x3, SAME zero padding, stride 1, no bias (lib.rs:204-216)
            {
                const int c = t & 31, pg = t >> 5;
                const float *dw = blk + B_DW;
                for (int p = pg; p < kCells; p += 8) {
                    const int y = p / kSide, x = p % kSide;
                    float acc = 0.0f;
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky) {
                        const int yy = y + ky - 1;
                        if (yy < 0 || yy >= kSide) continue;
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            const int xx = x + kx - 1;
                            if (xx < 0 || xx >= kSide) continue;
                            acc = fmaf(H0[(yy * kSide + xx) * kHStride + c], dw[(ky * 3 + kx) * kMid + c], acc);
                        }
                    }
                    H1[p * kHStride + c] = acc;
                }
            }
            __syncthreads();
            // conv1 pointwise 1x1 32 -> 32, bias, lrelu (lib.rs:232-255 + caller's activation1)
            gemm_n32<kMid, kHStride>(H1, blk + B_PW, blk + B_B1, H0, t);
            __syncthreads();
            // conv2: 1x1 32 -> 128, bias, + x, lrelu (lib.rs:432-450; network.rs:108-111)
            {
                const int tx = t & 31, ty = t >> 5;
                const float *W2 = blk + B_W2;
                float acc[11][4];
#pragma unroll
                for (int i = 0; i < 11; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
#pragma unroll 2
                for (int k = 0; k < kMid; k += 4) {
                    float4 w[4];
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) w[kk] = *reinterpret_cast<const float4 *>(W2 + (k + kk) * kCh + tx * 4);
#pragma unroll
                    for (int i = 0; i < 11; ++i) {
                        const int rr = min(ty + 8 * i, kCells - 1);
                        const float4 a = *reinterpret_cast<const float4 *>(H0 + rr * kHStride + k);
                        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            acc[i][0] = fmaf(av[kk], w[kk].x, acc[i][0]);
                            acc[i][1] = fmaf(av[kk], w[kk].y, acc[i][1]);
                            acc[i][2] = fmaf(av[kk], w[kk].z, acc[i][2]);
                            acc[i][3] = fmaf(av[kk], w[kk].w, acc[i][3]);
                        }
                    }
                }
                const float4 b = *reinterpret_cast<const float4 *>(blk + B_B2 + tx * 4);
#pragma unroll
                for (int i = 0; i < 11; ++i) {
                    const int rr = ty + 8 * i;
                    if (rr < kCells) {
                        float4 *xp = reinterpret_cast<float4 *>(X + rr * kXStride + tx * 4);
                        const float4 xr = *xp;
                        float4 o;
                        o.x = lrelu(acc[i][0] + b.x + xr.x);
                        o.y = lrelu(acc[i][1] + b.y + xr.y);
                        o.z = lrelu(acc[i][2] + b.z + xr.z);
                        o.w = lrelu(acc[i][3] + b.w + xr.w);
                        *xp = o;
                    }
                }
            }
            __syncthreads();
        }
        // ---- flatten NHWC: index = pixel*128 + channel (network.rs:127-137) ----
        {
            float *dst = act0 + (size_t)row * kFlat;
            for (int idx = t; idx < kCells * 32; idx += kTowerThreads) {
                const int pix = idx >> 5, c4 = (idx & 31) * 4;
                *reinterpret_cast<float4 *>(dst + pix * kCh + c4) = *reinterpret_cast<const float4 *>(X + pix * kXStride + c4);
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------
// C[M x N] = act(A[M x K] . W[K x N] + bias[N]); M = *n_req rounded up to the tile, N % 128 == 0,
// K % 16 == 0.  128x128x16 tiles, 256 threads, 8x8 outputs per thread, register double buffer.
// ---------------------------------------------------------------------------------------
constexpr int GM = 128, GN = 128, GK = 16, GPAD = 4;

__global__ void __launch_bounds__(256, 2)
    k_gemm(const float *__restrict__ A, const float *__restrict__ W, const float *__restrict__ bias, float *__restrict__ C,
           const uint32_t *n_req, int max_rows, int N, int K, int act) {
    __shared__ __align__(16) float As[2][GK][GM + GPAD];
    __shared__ __align__(16) float Bs[2][GK][GN];
    const int rows = (int)min(*n_req, (uint32_t)max_rows);
    const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
    if (m0 >= rows) return;
    const int t = threadIdx.x;
    const int tx = t & 15, ty = t >> 4;
    // global->smem mapping
    const int a_row = t >> 2, a_k = (t & 3) * 4;   // rows a_row, a_row+64; 4 consecutive k
    const int b_k = t >> 4, b_n = (t & 15) * 8;    // one k row, 8 consecutive n
    const float *Ap0 = A + (size_t)(m0 + a_row) * K + a_k;
    const float *Ap1 = A + (size_t)(m0 + a_row + 64) * K + a_k;
    const float *Bp = W + (size_t)b_k * N + n0 + b_n;

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

    float4 ra0 = *reinterpret_cast<const float4 *>(Ap0);
    float4 ra1 = *reinterpret_cast<const float4 *>(Ap1);
    float4 rb0 = *reinterpret_cast<const float4 *>(Bp);
    float4 rb1 = *reinterpret_cast<const float4 *>(Bp + 4);
    auto stage = [&](int buf) {
        As[buf][a_k + 0][a_row] = ra0.x; As[buf][a_k + 1][a_row] = ra0.y;
        As[buf][a_k + 2][a_row] = ra0.z; As[buf][a_k + 3][a_row] = ra0.w;
        As[buf][a_k + 0][a_row + 64] = ra1.x; As[buf][a_k + 1][a_row + 64] = ra1.y;
        As[buf][a_k + 2][a_row + 64] = ra1.z; As[buf][a_k + 3][a_row + 64] = ra1.w;
        *reinterpret_cast<float4 *>(&Bs[buf][b_k][b_n]) = rb0;
        *reinterpret_cast<float4 *>(&Bs[buf][b_k][b_n + 4]) = rb1;
    };
    stage(0);
    __syncthreads();
    const int nk = K / GK;
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) {
            const size_t ko = (size_t)(kt + 1) * GK;
            ra0 = *reinterpret_cast<const float4 *>(Ap0 + ko);
            ra1 = *reinterpret_cast<const float4 *>(Ap1 + ko);
            rb0 = *reinterpret_cast<const float4 *>(Bp + ko * N);
            rb1 = *reinterpret_cast<const float4 *>(Bp + ko * N + 4);
        }
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[buf][k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[buf][k][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kt + 1 < nk) stage(buf ^ 1);
        __syncthreads();
    }
    const float4 bb0 = *reinterpret_cast<const float4 *>(bias + n0 + tx * 4);
    const float4 bb1 = *reinterpret_cast<const float4 *>(bias + n0 + 64 + tx * 4);
    const float bvv[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            o[j] = acc[i][j] + bvv[j];
            if (act) o[j] = lrelu(o[j]);
        }
        float *cp = C + (size_t)row * N + n0;
        *reinterpret_cast<float4 *>(cp + tx * 4) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4 *>(cp + 64 + tx * 4) = make_float4(o[4], o[5], o[6], o[7]);
    }
}

// value = tanh(logit[81]); policy = softmax(logit[0..81)) (network.rs:188-247)
__global__ void k_heads(const float *logits, const uint32_t *n_req, int max_rows, float *P, float *V) {
    const int rows = (int)min(*n_req, (uint32_t)max_rows);
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float *l = logits + (size_t)row * 128;
    float v[3];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = lane + 32 * j;
        v[j] = c < kCells ? l[c] : -INFINITY;
        mx = fmaxf(mx, v[j]);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        v[j] = (lane + 32 * j) < kCells ? expf(v[j] - mx) : 0.0f;
        s += v[j];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float inv = 1.0f / s;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = lane + 32 * j;
        if (c < kCells) P[(size_t)row * kRow + c] = v[j] * inv;
    }
    if (lane == 0) V[row] = tanhf(l[kCells]);
}

// heads weight packing: [512][128] = {p_w[512][81] | v_w[512][1] | 0}
__global__ void k_pack_heads(const float *p_w, const float *p_b, const float *v_w, const float *v_b, float *hw, float *hb) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < kFc * 128) {
        const int k = idx >> 7, c = idx & 127;
        hw[idx] = c < kCells ? p_w[k * kCells + c] : (c == kCells ? v_w[k] : 0.0f);
    }
    if (idx < 128) hb[idx] = idx < kCells ? p_b[idx] : (idx == kCells ? v_b[0] : 0.0f);
}

// w = N(0,1) * scale (network-utils lib.rs:86-92); Box-Muller over the specified counter stream
__global__ void k_init_normal(float *w, long long n, float scale, uint64_t seed, uint32_t tensor) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r1 = rng_u32(seed ^ 0x5EED5EED5EEDull, tensor, (uint32_t)(2 * i));
    const uint32_t r2 = rng_u32(seed ^ 0x5EED5EED5EEDull, tensor, (uint32_t)(2 * i + 1));
    const float u1 = ((float)(r1 >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r2 >> 8) + 0.5f) * (1.0f / 16777216.0f);
    w[i] = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2) * scale;
}

void net_pack_heads(omk_ctx *c) {
    k_pack_heads<<<(kFc * 128 + 255) / 256, 256, 0, c->stream>>>(c->model->t[29], c->model->t[30], c->model->t[27], c->model->t[28],
                                                                  c->model->heads_w, c->model->heads_b);
    c->launches++;
}

static const long long kTensorLen[kNetTensors] = {
    384, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    (long long)kFlat * kFc, kFc, kFc * kFc, kFc, kFc, 1, kFc * kCells, kCells};

void launch_net_init_random(omk_ctx *c, uint64_t seed) {
    // He: 2/sqrt(fan_in); Xavier: 2/sqrt(fan_in+fan_out); depthwise fan_in = 3*3*32 (lib.rs:199-202)
    const float he3 = 2.0f / sqrtf(3.0f), he128 = 2.0f / sqrtf(128.0f), he288 = 2.0f / sqrtf(288.0f),
                he32 = 2.0f / sqrtf(32.0f), he_flat = 2.0f / sqrtf((float)kFlat), he512 = 2.0f / sqrtf(512.0f),
                xv = 2.0f / sqrtf(513.0f), xp = 2.0f / sqrtf(593.0f);
    float scale[kNetTensors] = {he3, 0, he128, 0, he288, he32, 0, he32, 0, he128, 0, he288, he32, 0, he32, 0,
                                he128, 0, he288, he32, 0, he32, 0, he_flat, 0, he512, 0, xv, 0, xp, 0};
    for (int i = 0; i < kNetTensors; ++i) {
        if (scale[i] == 0.0f) {
            cudaMemsetAsync(c->net.t[i], 0, sizeof(float) * kTensorLen[i], c->stream);
        } else {
            k_init_normal<<<(unsigned)((kTensorLen[i] + 255) / 256), 256, 0, c->stream>>>(c->net.t[i], kTensorLen[i], scale[i],
                                                                                          seed, (uint32_t)i);
            c->launches++;
        }
    }
}

// false: a launch, a tensor-map encode or an activation-buffer allocation failed -- ws.P / ws.V hold nothing the caller may
// use (the message went to stderr); callers must not run k_apply on them and return OMK_ERR_CUDA.
bool net_forward(omk_ctx *c, const float *images_dev, int max_rows) {
    cudaFuncSetAttribute(k_tower, cudaFuncAttributeMaxDynamicSharedMemorySize, kTowerSmemBytes);
    if (max_rows > c->ws.max_rows) max_rows = c->ws.max_rows;
    if (max_rows <= 0) return true;
    bool ok = true;
    TowerWeights tw;
    tw.conv_w = c->model->t[0];
    tw.conv_b = c->model->t[1];
    for (int r = 0; r < 3; ++r) {
        const int b = 2 + 7 * r;
        tw.w0[r] = c->model->t[b + 0]; tw.b0[r] = c->model->t[b + 1]; tw.dw[r] = c->model->t[b + 2]; tw.pw[r] = c->model->t[b + 3];
        tw.b1[r] = c->model->t[b + 4]; tw.w2[r] = c->model->t[b + 5]; tw.b2[r] = c->model->t[b + 6];
    }
    if (!ensure_activations(c, max_rows)) {
        fprintf(stderr, "omok_b200: activation workspace allocation failed (%d rows)\n", max_rows);
        return false;
    }
    const int tower_grid = max_rows < c->n_sms ? max_rows : c->n_sms;
    const int mt = (max_rows + GM - 1) / GM;
    const long long n0 = (long long)max_rows * kFlat, n1 = (long long)max_rows * kFc;
    // tower_mode / fc0_mode: 1 = tcgen05 3xFP16 kernels (the product path), 0 = fp32 CUDA-core kernels, kept only as an
    // in-library A/B check of each layer.  A mixed setting goes through an explicit conversion pass.
    bool sp = prof_begin(c, OMK_K_TOWER, 1);
    if (c->tower_mode == 1) {
        ok = launch_tower_f16(c, images_dev, max_rows) && ok;
        c->launches--;  // counted once below with the other network kernels
        if (c->fc0_mode == 0) launch_split16_to_f32(c, c->ws.act0_h16, c->ws.act0_l16, c->ws.act0, n0);
    } else {
        k_tower<<<tower_grid, kTowerThreads, kTowerSmemBytes, c->stream>>>(tw, c->ws.nn_in, images_dev, c->ws.n_req, max_rows,
                                                                          c->ws.act0);
        if (c->fc0_mode == 1) launch_f32_to_split16(c, c->ws.act0, c->ws.act0_h16, c->ws.act0_l16, n0);
    }
    prof_end(c, sp);
    sp = prof_begin(c, OMK_K_FC0, 1);
    if (c->fc0_mode == 1) {
        ok = launch_fc0_f16(c, max_rows) && ok;
        c->launches--;
    } else {
        k_gemm<<<dim3(kFc / GN, mt), 256, 0, c->stream>>>(c->ws.act0, c->model->t[23], c->model->t[24], c->ws.act1, c->ws.n_req,
                                                          max_rows, kFc, kFlat, 1);
        launch_f32_to_split16(c, c->ws.act1, c->ws.act1_h16, c->ws.act1_l16, n1);  // keeps debug buffer 9 meaningful
    }
    prof_end(c, sp);
    sp = prof_begin(c, OMK_K_FC1, 2);
    if (c->fc0_mode == 1) {
        ok = launch_fc1_f16(c, max_rows) && ok;
        c->launches--;
    } else {
        k_gemm<<<dim3(kFc / GN, mt), 256, 0, c->stream>>>(c->ws.act1, c->model->t[25], c->model->t[26], c->ws.act2, c->ws.n_req,
                                                          max_rows, kFc, kFc, 1);
    }
    prof_end(c, sp);
    sp = prof_begin(c, OMK_K_HEADS, 2);
    if (c->fc0_mode == 1) {  // heads GEMM + tanh / softmax in one tensor-core kernel
        ok = launch_heads_f16(c, max_rows) && ok;
    } else {
        k_gemm<<<dim3(1, mt), 256, 0, c->stream>>>(c->ws.act2, c->model->heads_w, c->model->heads_b, c->ws.logits, c->ws.n_req, max_rows,
                                                   128, kFc, 0);
        k_heads<<<(max_rows + 7) / 8, 256, 0, c->stream>>>(c->ws.logits, c->ws.n_req, max_rows, c->ws.P, c->ws.V);
        c->launches++;
    }
    prof_end(c, sp);
    c->launches += 3;  // tower, fc0, fc1 (launch_heads_f16 / the CUDA-core heads counted above)
    if (cudaPeekAtLastError() != cudaSuccess) {
        fprintf(stderr, "omok_b200: network forward: %s\n", cudaGetErrorString(cudaPeekAtLastError()));
        ok = false;
    }
    return ok;
}

}  // namespace omk
