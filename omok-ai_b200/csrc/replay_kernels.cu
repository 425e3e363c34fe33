// replay_kernels.cu -- the replay memory of the trainer (src/trainer.rs:27,206-352) on the device, next to the self-play
// driver that fills it.  Same rows, in the same order, as trainer.ReplayMemory fed with split_episodes one ply at a time:
// episodes in (ply of the final move, game id) order; within an episode the T original transitions, then the five
// symmetric copies of each transition, t-major, in AUGMENT_ORDER; value targets alternate backwards from the last ply's
// (1 for a win of its mover, 0 for a draw: +0.0 / -0.0 alternate as on the host); drop-oldest beyond the capacity.
//
//   staging  per game, up to 81 plies of (board u8[81], visit policy f32[81]) written at index sp_ply[g] when the ply is
//            recorded (k_rp_stage), plus the ply count
//   commit   one launch per ply on the replay stream, behind both search lanes' record of that ply (k_rp_commit)
//   rows     structure of arrays boards u8[cap][81], turns u8[cap], pi f32[cap][81], z f32[cap]; a ring addressed by the
//            absolute row number (rows added since the last reset) modulo the capacity
//   sampler  Floyd's sample without replacement on a specified random stream (k_rp_sample; DESIGN.md 4)
//   encode   gather + encode_nn_input (Player mode) straight into the trainer step's minibatch buffers (k_rp_gather)
#include "omk_internal.h"

namespace omk {

constexpr int kMaxPlies = kCells;  // a 9 x 9 game ends (at the latest in a draw) after 81 moves

struct SymTable {
    uint8_t p[5][kCells];
};
// dst[i*9 + j] = src[perm[i*9 + j]] of trainer.SYMMETRIES (src/utils.rs:1-64), in AUGMENT_ORDER (trainer.rs:223-315):
// rotate_90, rotate_180, rotate_270, flip_horizontal, flip_vertical
static constexpr SymTable make_sym_table() {
    SymTable t{};
    for (int i = 0; i < kSide; ++i)
        for (int j = 0; j < kSide; ++j) {
            const int k = i * kSide + j, r = kSide - 1;
            t.p[0][k] = (uint8_t)((r - j) * kSide + i);
            t.p[1][k] = (uint8_t)((r - i) * kSide + (r - j));
            t.p[2][k] = (uint8_t)(j * kSide + (r - i));
            t.p[3][k] = (uint8_t)(i * kSide + (r - j));
            t.p[4][k] = (uint8_t)((r - i) * kSide + j);
        }
    return t;
}
__constant__ SymTable c_sym = make_sym_table();

// the sampler's stream key: distinct from the Dirichlet noise's (omk_device.cuh, noise_gamma_cell)
constexpr uint64_t kReplaySamplerKey = 0x2545F4914F6CDD1Dull;

// ---- staging: one block per game of a search lane ----
__global__ void k_rp_stage(int g0, int n, const int32_t *__restrict__ ply, const uint8_t *__restrict__ boards,
                           const float *__restrict__ policy, uint8_t *__restrict__ stage_boards, float *__restrict__ stage_pi,
                           int32_t *__restrict__ stage_len) {
    const int i = blockIdx.x, g = g0 + i;
    if (i >= n) return;
    const int p = ply[g];
    if (p < 0 || p >= kMaxPlies) return;  // unreachable: a game has at most 81 plies
    const size_t dst = ((size_t)g * kMaxPlies + p) * kCells;
    for (int c = threadIdx.x; c < kCells; c += blockDim.x) {
        stage_boards[dst + c] = boards[(size_t)i * kCells + c];
        stage_pi[dst + c] = policy[(size_t)i * kCells + c];
    }
    if (threadIdx.x == 0) stage_len[g] = p + 1;
}

// ---- commit: the episodes that ended at this ply -> rows ----
// Every block scans the ply's statuses in game order (block-wide exclusive prefix sums of 6T rows and of finished games);
// block b writes the episodes whose rank in the ply is b modulo the grid.  The ring counters are read by every block at
// the start and advanced by the last block to finish (arrival counter, re-armed), so no block reads them half-updated.
constexpr int kCommitThreads = 256;

__device__ __forceinline__ void block_scan2(int a, int b, int *excl_a, int *excl_b, int *tot_a, int *tot_b, int2 *sh) {
    // inclusive warp scans, then the warps' totals
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int ia = a, ib = b;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int xa = __shfl_up_sync(0xffffffffu, ia, off), xb = __shfl_up_sync(0xffffffffu, ib, off);
        if (lane >= off) { ia += xa; ib += xb; }
    }
    if (lane == 31) sh[w] = make_int2(ia, ib);
    __syncthreads();
    int pa = 0, pb = 0, ta = 0, tb = 0;
    for (int k = 0; k < kCommitThreads / 32; ++k) {
        const int2 v = sh[k];
        if (k < w) { pa += v.x; pb += v.y; }
        ta += v.x;
        tb += v.y;
    }
    __syncthreads();  // sh is reused by the next call
    *excl_a = pa + ia - a;
    *excl_b = pb + ib - b;
    *tot_a = ta;
    *tot_b = tb;
}

__global__ void __launch_bounds__(kCommitThreads)
    k_rp_commit(int n, const int8_t *__restrict__ status, const int32_t *__restrict__ stage_len,
                const uint8_t *__restrict__ stage_boards, const float *__restrict__ stage_pi, ReplayRing ring,
                ReplayCounters *__restrict__ ctr) {
    __shared__ int2 sh_scan[kCommitThreads / 32];
    __shared__ int sh_game[kCommitThreads], sh_off[kCommitThreads];
    __shared__ int sh_count;
    __shared__ uint8_t sh_turn[kMaxPlies];
    __shared__ bool sh_last;
    const long long added0 = ctr->added, cap = ring.cap;
    auto finished_rows = [&](int g, int *fin) {
        *fin = 0;
        if (g >= n) return 0;
        const int st = status[g];
        if (st < kDraw || st > kWhiteWin) return 0;
        *fin = 1;
        return 6 * stage_len[g];
    };
    // pass 1: rows and episodes of the whole ply (the capacity rule keeps the LAST `cap` rows of the ring + this ply)
    long long total_rows = 0;
    int total_eps = 0;
    for (int base = 0; base < n; base += kCommitThreads) {
        int fin;
        const int rows = finished_rows(base + threadIdx.x, &fin);
        int ea, eb, ta, tb;
        block_scan2(rows, fin, &ea, &eb, &ta, &tb, sh_scan);
        total_rows += ta;
        total_eps += tb;
    }
    const long long keep_from = added0 + total_rows - cap;  // absolute rows below this one are dropped by the ply's end
    // pass 2: write this block's episodes
    long long run_rows = 0;
    int run_eps = 0;
    for (int base = 0; base < n && total_eps > 0; base += kCommitThreads) {
        const int g = base + threadIdx.x;
        int fin;
        const int rows = finished_rows(g, &fin);
        int ea, eb, ta, tb;
        block_scan2(rows, fin, &ea, &eb, &ta, &tb, sh_scan);
        if (threadIdx.x == 0) sh_count = 0;
        __syncthreads();
        if (fin && (run_eps + eb) % (int)gridDim.x == (int)blockIdx.x) {
            const int k = atomicAdd(&sh_count, 1);
            sh_game[k] = g;
            sh_off[k] = ea;
        }
        __syncthreads();
        const int count = sh_count;
        for (int k = 0; k < count; ++k) {
            const int gk = sh_game[k], T = stage_len[gk];
            const float fz = status[gk] == kDraw ? 0.0f : 1.0f;
            const long long first = added0 + run_rows + sh_off[k];  // absolute row of the episode's first original
            // rows r < skip are dropped by the ply's end; row r lives at (phys0 + r) % cap (32-bit: cap < 2^31, r < 486)
            const int skip = first >= keep_from ? 0 : (int)min(keep_from - first, (long long)kMaxPlies * 6);
            const uint32_t phys0 = (uint32_t)(first % cap), ucap = (uint32_t)cap;
            const uint8_t *sb = stage_boards + (size_t)gk * kMaxPlies * kCells;
            const float *sp = stage_pi + (size_t)gk * kMaxPlies * kCells;
            for (int t = threadIdx.x; t < T; t += blockDim.x) {  // turn from the stone counts (0 = Black to move)
                int nb = 0, nw = 0;
                for (int c = 0; c < kCells; ++c) {
                    const uint8_t v = sb[t * kCells + c];
                    nb += v == 1;
                    nw += v == 2;
                }
                sh_turn[t] = nb != nw ? 1 : 0;
            }
            __syncthreads();
            const int R = 6 * T;
            for (int r = skip + threadIdx.x; r < R; r += blockDim.x) {
                const int t = r < T ? r : (r - T) / 5;
                const size_t phys = (phys0 + (uint32_t)r) % ucap;
                ring.turns[phys] = sh_turn[t];
                ring.z[phys] = ((T - 1 - t) & 1) ? -fz : fz;
            }
            for (int e = skip * kCells + threadIdx.x; e < R * kCells; e += blockDim.x) {
                const int r = e / kCells, c = e - r * kCells;
                int t, src = c;
                if (r < T) {
                    t = r;
                } else {
                    t = (r - T) / 5;
                    src = c_sym.p[(r - T) % 5][c];
                }
                const size_t phys = (phys0 + (uint32_t)r) % ucap;
                ring.boards[phys * kCells + c] = sb[t * kCells + src];
                ring.pi[phys * kCells + c] = sp[t * kCells + src];
            }
            __syncthreads();  // sh_turn is rewritten by the next episode
        }
        run_rows += ta;
        run_eps += tb;
    }
    // the last block to finish advances the ring
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) sh_last = atomicAdd(&ctr->done, 1u) == gridDim.x - 1u;
    __syncthreads();
    if (!sh_last || threadIdx.x != 0) return;
    const long long len = ctr->len + total_rows;
    ctr->added = added0 + total_rows;
    ctr->len = len < cap ? len : cap;
    ctr->episodes += total_eps;
    ctr->done = 0u;
}

// ---- sampler: one warp per step ----
// Floyd: for j in len-m .. len-1 { t = below(j + 1); append j if t was already chosen, else t }; stream keyed by
// (mix64(seed ^ kReplaySamplerKey), stream = step index, counter from 0); below = rand's sample_single (rng_below).
__global__ void k_rp_sample(uint64_t key, long long first_step, int steps, long long len, int m, int64_t *__restrict__ rows) {
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (s >= steps) return;
    int64_t *out = rows + (size_t)s * m;
    const uint32_t stream = (uint32_t)(first_step + s);
    uint32_t counter = 0;
    for (int k = 0; k < m; ++k) {
        const long long j = len - m + k;
        long long t = 0;
        if (lane == 0) t = rng_below(key, stream, counter, (uint32_t)(j + 1));
        t = __shfl_sync(0xffffffffu, t, 0);
        bool seen = false;
        for (int i = lane; i < k; i += 32) seen |= out[i] == t;
        const bool dup = __any_sync(0xffffffffu, seen);
        if (lane == 0) out[k] = dup ? j : t;
        __syncwarp();
    }
}

// ---- gather + encode: one block per minibatch row ----
__global__ void k_rp_gather(const int64_t *__restrict__ rows, int m, ReplayRing ring, long long base, float *__restrict__ img,
                            float *__restrict__ pi, float *__restrict__ z) {
    const int i = blockIdx.x;
    if (i >= m) return;
    const size_t phys = (size_t)((base + rows[i]) % ring.cap);
    const uint8_t turn = ring.turns[phys];
    const uint8_t *b = ring.boards + phys * kCells;
    // encode_nn_input, EnvTurnMode::Player: (cell, {side to move, other side}) pairs, then the Black-to-move plane
    const uint8_t first = turn == 0 ? 1 : 2;
    for (int f = threadIdx.x; f < 243; f += blockDim.x) {
        float v;
        if (f >= 2 * kCells) v = turn == 0 ? 1.0f : 0.0f;
        else {
            const uint8_t cell = b[f >> 1];
            v = cell != 0 && ((f & 1) == 0) == (cell == first) ? 1.0f : 0.0f;
        }
        img[(size_t)i * 243 + f] = v;
    }
    for (int c = threadIdx.x; c < kCells; c += blockDim.x) pi[(size_t)i * kCells + c] = ring.pi[phys * kCells + c];
    if (threadIdx.x == 0) z[i] = ring.z[phys];
}

// ---- omk_replay_get: logical rows -> host layout ----
__global__ void k_rp_get(const int64_t *__restrict__ rows, int n, ReplayRing ring, long long base, uint8_t *__restrict__ boards,
                         uint8_t *__restrict__ turns, float *__restrict__ pi, float *__restrict__ z) {
    const int i = blockIdx.x;
    if (i >= n) return;
    const size_t phys = (size_t)((base + rows[i]) % ring.cap);
    for (int c = threadIdx.x; c < kCells; c += blockDim.x) {
        boards[(size_t)i * kCells + c] = ring.boards[phys * kCells + c];
        pi[(size_t)i * kCells + c] = ring.pi[phys * kCells + c];
    }
    if (threadIdx.x == 0) {
        turns[i] = ring.turns[phys];
        z[i] = ring.z[phys];
    }
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
void launch_rp_stage(omk_ctx *c, int g0, int n, const uint8_t *boards, const float *policy) {
    if (n <= 0) return;
    k_rp_stage<<<n, 96, 0, c->stream>>>(g0, n, c->sp_ply, boards, policy, c->rp.stage.boards, c->rp.stage.pi, c->rp.stage.len);
    c->launches++;
}
void launch_rp_commit(omk_ctx *c, int n, const int8_t *status) {
    const int blocks = n < c->n_sms ? n : c->n_sms;
    k_rp_commit<<<blocks, kCommitThreads, 0, c->rp.stream>>>(n, status, c->rp.stage.len, c->rp.stage.boards, c->rp.stage.pi,
                                                             c->rp.ring.view(), c->rp.counters);
    c->launches++;
}
void launch_rp_sample(omk_ctx *c, uint64_t seed, long long first_step, int steps, long long len, int m, int64_t *rows) {
    const int warps = 4;
    k_rp_sample<<<(steps + warps - 1) / warps, 32 * warps, 0, c->stream>>>(mix64(seed ^ kReplaySamplerKey), first_step, steps, len,
                                                                           m, rows);
    c->launches++;
}
void launch_rp_gather(omk_ctx *c, const int64_t *rows, int m, float *img, float *pi, float *z) {
    k_rp_gather<<<m, 96, 0, c->stream>>>(rows, m, c->rp.ring.view(), c->rp.added - c->rp.len, img, pi, z);
    c->launches++;
}
void launch_rp_get(omk_ctx *c, const int64_t *rows, int n, uint8_t *boards, uint8_t *turns, float *pi, float *z) {
    k_rp_get<<<n, 96, 0, c->stream>>>(rows, n, c->rp.ring.view(), c->rp.added - c->rp.len, boards, turns, pi, z);
    c->launches++;
}

}  // namespace omk
