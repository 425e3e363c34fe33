// omk_device.cuh -- shared device-side definitions for libomok_b200 (sm_100a only).
//
// HBM layout (see DESIGN.md "Data layout"):
//   env pool   : 32-byte packed record per board  {black[3], white[3], meta, pad}
//   tree pool  : per tree a 64-byte TreeHdr and `capacity_nodes` node records of
//                1408 bytes = {48 B header + pad | policy[96] f32 | edge_n[96] u32 |
//                edge_w[96] f32 | child[96] u16}.  Statistics live on EDGES, stored at
//                the parent and indexed by ACTION, so a PUCT scan of a node is three
//                coalesced 324-byte row reads with no gather.  A child's prior is the
//                parent's policy entry (the reference keeps child.p == parent.policy[a]
//                at all times: node.rs:76, parallel_mcts_executor.rs:70-75,256-261), and
//                creation order == node-id order, so "last maximum wins" (max_by) is
//                "largest child id among the maxima".
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace omk {

constexpr int kCells = 81;
constexpr int kSide = 9;
constexpr int kRow = 96;  // padded row length of per-action arrays (3 x 128 B lines)
constexpr uint32_t kNoNode = 0xFFFFu;
constexpr float kF32Eps = 1.1920929e-7f;  // f32::EPSILON

// status codes (environment/src/lib.rs:45-51)
constexpr int kInProgress = 0, kDraw = 1, kBlackWin = 2, kWhiteWin = 3;

// ---- node record ----
constexpr int kNodeBytes = 1408;
constexpr int kOffPolicy = 64;
constexpr int kOffEdgeN = 448;
constexpr int kOffEdgeW = 832;
constexpr int kOffChild = 1216;

// header words: 0-2 black, 3-5 white, 6-8 childmask, 9 = parent | action<<16 | status<<24,
// 10 = legal | turn<<8 | has_policy<<16
struct NodeHdr {
    uint32_t black[3], white[3], cmask[3];
    uint32_t parent, action, status, legal, turn, has_policy;
};

struct __align__(16) TreeHdr {
    uint32_t n_nodes;      // bump pointer == live nodes after compaction
    uint32_t root_n;       // root.n (mcts/src/node.rs:20)
    float root_w;          // root.w
    float root_p;          // root.p (1.0 for a fresh tree, mcts/src/lib.rs:27)
    uint32_t rng_counter;  // position in the tree's random stream
    uint32_t stream;       // stream id
    uint32_t noise_epoch;  // Dirichlet applications so far
    uint32_t error;        // sticky: 1 = node capacity exceeded
    uint32_t sims_lo, sims_hi;
    uint32_t pad[6];
};
static_assert(sizeof(TreeHdr) == 64, "TreeHdr is 64 bytes");

struct __align__(16) NNIn {  // one evaluator request: packed board, 32 bytes
    uint32_t black[3], white[3];
    uint32_t meta;  // bit0 turn, bit1 opponent-mode
    uint32_t pad;
};

struct __align__(16) EnvRec {  // env pool record, 32 bytes
    uint32_t black[3], white[3];
    uint32_t meta;  // bit0 turn, bits 8..15 legal_move_count
    uint32_t pad;
};

__device__ __forceinline__ uint8_t *node_ptr(uint8_t *tree_nodes, uint32_t id) {
    return tree_nodes + (size_t)id * kNodeBytes;
}
__device__ __forceinline__ float *node_policy(uint8_t *n) { return reinterpret_cast<float *>(n + kOffPolicy); }
__device__ __forceinline__ uint32_t *node_edge_n(uint8_t *n) { return reinterpret_cast<uint32_t *>(n + kOffEdgeN); }
__device__ __forceinline__ float *node_edge_w(uint8_t *n) { return reinterpret_cast<float *>(n + kOffEdgeW); }
__device__ __forceinline__ uint16_t *node_child(uint8_t *n) { return reinterpret_cast<uint16_t *>(n + kOffChild); }

__device__ __forceinline__ NodeHdr load_hdr(const uint8_t *n) {
    const uint4 *q = reinterpret_cast<const uint4 *>(n);
    const uint4 a = q[0], b = q[1], c = q[2];
    NodeHdr h;
    h.black[0] = a.x; h.black[1] = a.y; h.black[2] = a.z;
    h.white[0] = a.w; h.white[1] = b.x; h.white[2] = b.y;
    h.cmask[0] = b.z; h.cmask[1] = b.w; h.cmask[2] = c.x;
    h.parent = c.y & 0xFFFFu; h.action = (c.y >> 16) & 0xFFu; h.status = c.y >> 24;
    h.legal = c.z & 0xFFu; h.turn = (c.z >> 8) & 0xFFu; h.has_policy = (c.z >> 16) & 0xFFu;
    return h;
}
__device__ __forceinline__ void store_hdr(uint8_t *n, const NodeHdr &h) {
    uint4 *q = reinterpret_cast<uint4 *>(n);
    q[0] = make_uint4(h.black[0], h.black[1], h.black[2], h.white[0]);
    q[1] = make_uint4(h.white[1], h.white[2], h.cmask[0], h.cmask[1]);
    q[2] = make_uint4(h.cmask[2], h.parent | (h.action << 16) | (h.status << 24),
                      h.legal | (h.turn << 8) | (h.has_policy << 16), 0u);
}

// ---- 81-bit masks in three words ----
__device__ __forceinline__ uint32_t sel3(uint32_t w0, uint32_t w1, uint32_t w2, int word) {
    return word == 0 ? w0 : (word == 1 ? w1 : w2);
}
__device__ __forceinline__ bool bit81(const uint32_t *m, int i) { return (sel3(m[0], m[1], m[2], i >> 5) >> (i & 31)) & 1u; }
__device__ __forceinline__ void set81(uint32_t *m, int i) {
    const uint32_t b = 1u << (i & 31);
    if ((i >> 5) == 0) m[0] |= b; else if ((i >> 5) == 1) m[1] |= b; else m[2] |= b;
}
__device__ __forceinline__ int popc81(const uint32_t *m) { return __popc(m[0]) + __popc(m[1]) + __popc(m[2] & 0x1FFFFu); }
// index of the r-th (0-based) set bit, ascending
__device__ __forceinline__ int nth_set_bit32(uint32_t w, int r) {
    for (int i = 0; i < r; ++i) w &= w - 1;
    return __ffs(w) - 1;
}
__device__ __forceinline__ int nth_set81(const uint32_t *m, int r) {
    const int c0 = __popc(m[0]), c1 = __popc(m[1]);
    if (r < c0) return nth_set_bit32(m[0], r);
    if (r < c0 + c1) return 32 + nth_set_bit32(m[1], r - c0);
    return 64 + nth_set_bit32(m[2], r - c0 - c1);
}

// f32::total_cmp order key
__device__ __forceinline__ int32_t total_order_key(float f) {
    const int32_t b = __float_as_int(f);
    return b ^ (int32_t)((uint32_t)(b >> 31) >> 1);
}

// ---- specified random stream (DESIGN.md "Random stream"); the CPU checker implements the same spec ----
constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ull;
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint32_t rng_u32(uint64_t seed, uint32_t stream, uint32_t counter) {
    const uint64_t k = mix64(seed + kGolden * ((uint64_t)stream + 1));
    return (uint32_t)(mix64(k + kGolden * ((uint64_t)counter + 1)) >> 32);
}
// the naive player's random moves run on the key mix64(seed ^ kNaiveKey) (eval_kernels.cu)
constexpr uint64_t kNaiveKey = 0xA0761D6478BD642Full;
// rand 0.8.5 UniformInt::<u32>::sample_single (widening multiply + conservative zone)
__device__ __forceinline__ uint32_t rng_below(uint64_t seed, uint32_t stream, uint32_t &counter, uint32_t bound) {
    const uint32_t zone = (bound << __clz(bound)) - 1u;
    for (;;) {
        const uint32_t v = rng_u32(seed, stream, counter++);
        const uint64_t m = (uint64_t)v * (uint64_t)bound;
        if ((uint32_t)m <= zone) return (uint32_t)(m >> 32);
    }
}

// ---- deterministic double-precision elementary functions (no fma, IEEE ops only) ----
__device__ __forceinline__ double det_log(double x) {
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    int e = (int)((b >> 52) & 0x7ff) - 1023;
    b = (b & 0x000fffffffffffffull) | 0x3ff0000000000000ull;
    double m = __longlong_as_double((long long)b);
    if (m > 1.4142135623730951) {
        m = __dmul_rn(m, 0.5);
        e += 1;
    }
    const double s = __ddiv_rn(__dsub_rn(m, 1.0), __dadd_rn(m, 1.0));
    const double s2 = __dmul_rn(s, s);
    double acc = __ddiv_rn(1.0, 25.0);
    for (int k = 23; k >= 1; k -= 2) acc = __dadd_rn(__dmul_rn(acc, s2), __ddiv_rn(1.0, (double)k));
    const double logm = __dmul_rn(__dmul_rn(2.0, s), acc);
    return __dadd_rn(__dmul_rn((double)e, 0.6931471805599453), logm);
}
__device__ __forceinline__ double det_exp(double x) {
    if (x < -745.0) return 0.0;
    if (x > 709.0) return __longlong_as_double(0x7ff0000000000000ll);
    const double kf = floor(__dadd_rn(__dmul_rn(x, 1.4426950408889634), 0.5));
    const int k = (int)kf;
    const double r = __dsub_rn(__dsub_rn(x, __dmul_rn(kf, 6.93147180369123816490e-01)),
                               __dmul_rn(kf, 1.90821492927058770002e-10));
    const double inv_fact[14] = {1.0, 1.0, 1.0 / 2.0, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0, 1.0 / 720.0,
                                 1.0 / 5040.0, 1.0 / 40320.0, 1.0 / 362880.0, 1.0 / 3628800.0,
                                 1.0 / 39916800.0, 1.0 / 479001600.0, 1.0 / 6227020800.0};
    double acc = 1.0 / 87178291200.0;
#pragma unroll
    for (int i = 13; i >= 0; --i) acc = __dadd_rn(__dmul_rn(acc, r), inv_fact[i]);
    const int k1 = k / 2, k2 = k - k1;
    const double f1 = __longlong_as_double((long long)(k1 + 1023) << 52);
    const double f2 = __longlong_as_double((long long)(k2 + 1023) << 52);
    return __dmul_rn(__dmul_rn(acc, f1), f2);
}

// ---- Dirichlet noise: Gamma(alpha,1) for one cell from its own sub-stream ----
struct NoiseRng {
    uint64_t seed;
    uint32_t stream, base, j;
    __device__ __forceinline__ double unif() {
        const uint32_t r = rng_u32(seed, stream, base + (j++));
        return __dmul_rn(__dadd_rn((double)r, 0.5), 2.3283064365386963e-10);
    }
    __device__ double normal() {
        for (;;) {
            const double u = __dsub_rn(__dmul_rn(2.0, unif()), 1.0);
            const double v = __dsub_rn(__dmul_rn(2.0, unif()), 1.0);
            const double s = __dadd_rn(__dmul_rn(u, u), __dmul_rn(v, v));
            if (s >= 1.0 || s == 0.0) continue;
            return __dmul_rn(u, __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, det_log(s)), s)));
        }
    }
    __device__ double gamma_large(double shape) {
        const double d = __dsub_rn(shape, 1.0 / 3.0);
        const double c = __ddiv_rn(1.0, __dsqrt_rn(__dmul_rn(9.0, d)));
        for (;;) {
            const double x = normal();
            const double vc = __dadd_rn(1.0, __dmul_rn(c, x));
            if (vc <= 0.0) continue;
            const double v = __dmul_rn(__dmul_rn(vc, vc), vc);
            const double u = unif();
            const double x2 = __dmul_rn(x, x);
            if (u < __dsub_rn(1.0, __dmul_rn(__dmul_rn(0.0331, x2), x2))) return __dmul_rn(d, v);
            const double rhs = __dadd_rn(__dmul_rn(0.5, x2), __dmul_rn(d, __dadd_rn(__dsub_rn(1.0, v), det_log(v))));
            if (det_log(u) < rhs) return __dmul_rn(d, v);
        }
    }
    __device__ double gamma(double shape) {
        if (shape < 1.0) {
            const double u = unif();
            const double g = gamma_large(__dadd_rn(shape, 1.0));
            return __dmul_rn(g, det_exp(__ddiv_rn(det_log(u), shape)));
        }
        return gamma_large(shape);
    }
};
__device__ __forceinline__ float noise_gamma_cell(uint64_t seed, uint32_t stream, uint32_t epoch, int cell, float alpha) {
    NoiseRng g{mix64(seed ^ 0xD1B54A32D192ED03ull), stream, (epoch << 16) + ((uint32_t)cell << 9), 0u};
    return (float)g.gamma((double)alpha);
}

// ---- exact hash evaluator (OMK_EVAL_HASH); the CPU checker implements the same spec ----
__device__ __forceinline__ uint64_t hash_board(const uint32_t *black, const uint32_t *white, uint32_t turn, uint32_t opp) {
    uint64_t h = 0x243F6A8885A308D3ull;
    h = mix64(h ^ ((uint64_t)black[0] | ((uint64_t)black[1] << 32)));
    h = mix64(h ^ ((uint64_t)black[2] | ((uint64_t)white[0] << 32)));
    h = mix64(h ^ ((uint64_t)white[1] | ((uint64_t)white[2] << 32)));
    h = mix64(h ^ ((uint64_t)turn | ((uint64_t)opp << 1)));
    return h;
}
__device__ __forceinline__ float hash_policy(uint64_t h, int a) {
    return __fmul_rn((float)((uint32_t)(mix64(h + kGolden * (uint64_t)(a + 1)) >> 40) + 1u), 5.9604644775390625e-08f);
}
__device__ __forceinline__ float hash_value(uint64_t h) {
    return __fsub_rn(__fmul_rn((float)(uint32_t)(mix64(h + kGolden * 82ull) >> 40), 1.1920928955078125e-07f), 1.0f);
}

// ---- five-in-a-row (environment/src/lib.rs:115-159) ----
// Scalar form (one thread owns the board): run length through `idx` along (dx,dy),
// scanning at most 5 cells each way, stopping at the edge or a non-mover cell.
__device__ __forceinline__ int run_through(const uint32_t *s, int x0, int y0, int dx, int dy) {
    int count = 1;
#pragma unroll
    for (int sgn = -1; sgn <= 1; sgn += 2) {
#pragma unroll
        for (int k = 1; k <= 5; ++k) {
            const int x = x0 + sgn * dx * k, y = y0 + sgn * dy * k;
            if (x < 0 || x >= kSide || y < 0 || y >= kSide) break;
            if (!bit81(s, y * kSide + x)) break;
            ++count;
        }
    }
    return count;
}
__device__ __forceinline__ bool makes_five_scalar(const uint32_t *s, int idx) {
    const int x0 = idx % kSide, y0 = idx / kSide;
    return run_through(s, x0, y0, 1, 0) == 5 || run_through(s, x0, y0, 0, 1) == 5 ||
           run_through(s, x0, y0, 1, 1) == 5 || run_through(s, x0, y0, 1, -1) == 5;
}
// Warp form (the warp owns the board, `s` uniform across lanes): lanes 0..19 each test
// one (axis, side, step) cell; one ballot per axis pair yields all eight run lengths.
__device__ __forceinline__ bool makes_five_warp(const uint32_t *s, int idx, int lane) {
    const int x0 = idx % kSide, y0 = idx / kSide;
    bool five = false;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        const int axis = pass * 2 + (lane >= 10 ? 1 : 0);        // 0:(1,0) 1:(0,1) 2:(1,1) 3:(1,-1)
        const int side = ((lane % 10) >= 5) ? 1 : -1;
        const int k = lane % 5 + 1;
        const int dx = (axis == 1) ? 0 : 1;
        const int dy = (axis == 0) ? 0 : (axis == 3 ? -1 : 1);
        const int x = x0 + side * dx * k, y = y0 + side * dy * k;
        bool on = false;
        if (lane < 20 && x >= 0 && x < kSide && y >= 0 && y < kSide) on = bit81(s, y * kSide + x);
        const uint32_t b = __ballot_sync(0xffffffffu, on);
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const uint32_t neg = (b >> (a * 10)) & 31u, pos = (b >> (a * 10 + 5)) & 31u;
            const int cn = __ffs(~neg) - 1, cp = __ffs(~pos) - 1;  // consecutive ones from step 1
            five |= (1 + cn + cp) == 5;
        }
    }
    return five;
}

// The 243-float memory image of encode_nn_input (encoder.rs:22-43): floats [0,162) are
// encode_board's (cell, plane) pairs with the perspective side in plane 0, floats [162,243) the
// turn plane.  TensorFlow later reads the slot as [9,9,3]; the network kernels do the same.
__device__ __forceinline__ float image_value(const uint32_t *black, const uint32_t *white, uint32_t turn, uint32_t opp,
                                             int f) {
    if (f >= 2 * kCells) return turn == 0 ? 1.0f : 0.0f;
    const int cell = f >> 1, off = f & 1;
    const uint32_t persp = turn ^ opp;              // EnvTurnMode::Opponent flips the perspective
    const int black_off = persp == 0 ? 0 : 1;
    return (off == black_off ? bit81(black, cell) : bit81(white, cell)) ? 1.0f : 0.0f;
}


}  // namespace omk
