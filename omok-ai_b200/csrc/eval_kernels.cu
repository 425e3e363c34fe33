// eval_kernels.cu -- the trainer's evaluation against the naive player (src/trainer.rs:487-603) on the device: the naive
// player's move (:506-537) and the bookkeeping omk_eval_naive runs after every half-move; the same bookkeeping for the
// arena between the network and the opponent (omk_match, benchmark/src/main.rs:14-108), and for a round-robin of that arena
// over up to kModelSlots models, optionally with the naive player as participant 0 (omk_tournament, omk_tournament_naive).
#include "omk_internal.h"

namespace omk {

constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kNaiveWarps = 4;
constexpr int kAdvanceThreads = 1024;

// The naive player's rule (DESIGN.md 4) for one position, the warp owning it: the first empty cell, ascending, where
// place_stone is terminal for the mover or, on the same board with the turn flipped, for the opponent; else
// legal[below(legal_count)] on the stream (key, stream, counter from 0).  A forced move draws nothing.  out_status (may be
// null): place_stone's result for the move on this board (OMK_NONE when there is none).
__device__ __forceinline__ void naive_pick(const uint32_t *black, const uint32_t *white, uint32_t turn, uint64_t key, uint32_t stream,
                                           int lane, int32_t *out_action, uint8_t *out_forced, int8_t *out_status) {
    uint32_t empty[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) empty[k] = ~(black[k] | white[k]);
    empty[2] &= 0x1FFFFu;
    const int legal = popc81(empty);
    const uint32_t *mine = turn == 0 ? black : white, *theirs = turn == 0 ? white : black;
    uint32_t hit[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int a = lane + 32 * j;
        bool ends = false;
        if (a < kCells && bit81(empty, a)) {
            if (legal == 1) {
                ends = true;  // the last empty cell: Draw (or a win) for either side
            } else {
                uint32_t s[3] = {mine[0], mine[1], mine[2]}, o[3] = {theirs[0], theirs[1], theirs[2]};
                set81(s, a);
                set81(o, a);
                ends = makes_five_scalar(s, a) || makes_five_scalar(o, a);
            }
        }
        hit[j] = __ballot_sync(kFullMask, ends);
    }
    if (lane != 0) return;
    int action = OMK_NONE;
    uint8_t forced = 0;
    if (hit[0] | hit[1] | hit[2]) {
        action = hit[0] ? __ffs(hit[0]) - 1 : (hit[1] ? 32 + __ffs(hit[1]) - 1 : 64 + __ffs(hit[2]) - 1);
        forced = 1;
    } else if (legal > 0) {
        uint32_t counter = 0;
        action = nth_set81(empty, (int)rng_below(key, stream, counter, (uint32_t)legal));
    }
    *out_action = action;
    if (out_forced) *out_forced = forced;
    if (out_status) {
        int status = OMK_NONE;
        if (action != OMK_NONE) {
            uint32_t s[3] = {mine[0], mine[1], mine[2]};
            set81(s, action);
            status = makes_five_scalar(s, action) ? (turn == 0 ? kBlackWin : kWhiteWin) : (legal == 1 ? kDraw : kInProgress);
        }
        *out_status = (int8_t)status;
    }
}

// One warp per position.  Positions come either as cells + turns (omk_naive_move; stream = streams[i] or i) or as the
// root nodes of trees ids[i]: omk_eval_naive's (game g = ids[i] - first_tree, stream = g * 81 + ply[g]), or, with ply null,
// the opponents' trees of omk_tournament_naive (tree first_tree + 4 * pairs * p + 2 * pairs + g of pairing p holds game g,
// stream = g * 81 + half; every live game of a pairing has played `half` moves).
struct NaiveArgs {
    const uint8_t *boards, *turns;  // [n][81], [n]; nullptr: the tree roots below
    const uint32_t *streams;
    const int32_t *ids;
    const uint8_t *nodes;
    int cap_nodes, first_tree;
    const int32_t *ply;
    int pairs, half;
    int n;
    uint64_t key;
    int32_t *actions;
    uint8_t *forced;
    int8_t *status;  // [n] place_stone's result of each move (may be null)
};

__global__ void __launch_bounds__(kNaiveWarps * 32) k_naive_move(NaiveArgs a) {
    const int i = blockIdx.x * kNaiveWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= a.n) return;
    uint32_t black[3], white[3], turn, stream;
    if (a.boards) {
        const uint8_t *b = a.boards + (size_t)i * kCells;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int c = lane + 32 * j;
            const uint8_t v = c < kCells ? b[c] : 0;
            black[j] = __ballot_sync(kFullMask, v == 1);
            white[j] = __ballot_sync(kFullMask, v == 2);
        }
        turn = a.turns[i];
        stream = a.streams ? a.streams[i] : (uint32_t)i;
    } else {
        const int tree = a.ids[i];
        const NodeHdr h = load_hdr(a.nodes + (size_t)tree * (size_t)a.cap_nodes * kNodeBytes);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            black[k] = h.black[k];
            white[k] = h.white[k];
        }
        turn = h.turn;
        if (a.ply) {
            const int g = tree - a.first_tree;
            stream = (uint32_t)(g * kCells + a.ply[g]);
        } else {
            const int g = (tree - a.first_tree) % (4 * a.pairs) - 2 * a.pairs;
            stream = (uint32_t)(g * kCells + a.half);
        }
    }
    naive_pick(black, white, turn, a.key, stream, lane, a.actions + i, a.forced ? a.forced + i : nullptr,
               a.status ? a.status + i : nullptr);
}

// A fresh evaluation: live list = every game's tree, no move played, nothing tallied.
__global__ void k_eval_init(int episodes, int first_tree, int32_t *ids, int32_t *ply, int8_t *moves, int8_t *final_status,
                            int32_t *counters) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < episodes * kCells) moves[t] = -1;
    if (t < episodes) {
        ids[t] = first_tree + t;
        ply[t] = 0;
        final_status[t] = kInProgress;
    }
    if (t < 4) counters[t] = 0;
}

// After a half-move's k_play on the live trees ids[0..n): append each game's move to its record, tally and record the
// games that ended, and compact the live list in place, stably (ascending game order is kept).  One block.
// counters = {BlackWin, WhiteWin, Draw, live count}.
__global__ void __launch_bounds__(kAdvanceThreads) k_eval_advance(int32_t *ids, int n, const int32_t *actions, const int8_t *status,
                                                                  int first_tree, int32_t *ply, int8_t *moves, int8_t *final_status,
                                                                  int32_t *counters, uint32_t *dev_error) {
    __shared__ int warp_kept[kAdvanceThreads / 32];
    __shared__ int kept_before;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) kept_before = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += kAdvanceThreads) {
        const int i = c0 + threadIdx.x;
        bool keep = false;
        int32_t id = 0;
        if (i < n) {
            id = ids[i];
            const int g = id - first_tree;
            const int st = status[i];
            moves[(size_t)g * kCells + ply[g]] = (int8_t)actions[i];
            ply[g] += 1;
            if (st == kInProgress) {
                keep = true;
            } else if (st == kDraw || st == kBlackWin || st == kWhiteWin) {
                final_status[g] = (int8_t)st;
                atomicAdd(&counters[st == kBlackWin ? 0 : (st == kWhiteWin ? 1 : 2)], 1);
            } else {
                atomicOr(dev_error, 8u);  // Option::None: the move was refused -- the game could never end
            }
        }
        const uint32_t b = __ballot_sync(kFullMask, keep);
        if (lane == 0) warp_kept[warp] = __popc(b);
        __syncthreads();  // every id of this chunk has been read before any is overwritten
        int dst = kept_before + __popc(b & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) dst += warp_kept[w];
        if (keep) ids[dst] = id;
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < kAdvanceThreads / 32; ++w) kept_before += warp_kept[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) counters[3] = kept_before;
}

// A fresh match: tree k of the 4 * pairs is first_tree + k, laid out [model][leg][pairs] (network 0, opponent 1), so game j
// (leg j / pairs) has the network's tree first_tree + j and the opponent's first_tree + 2 * pairs + j; both use stream j % pairs.
__global__ void k_match_init(int pairs, int first_tree, int32_t *ids, uint32_t *streams, int8_t *moves, int8_t *final_status,
                             int32_t *counters) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int games = 2 * pairs;
    if (t < games * kCells) moves[t] = -1;
    if (t < 2 * games) ids[t] = first_tree + t;
    if (t < games) {
        streams[t] = (uint32_t)(t % pairs);
        final_status[t] = kInProgress;
    }
    if (t < 8) counters[t] = 0;
}

// After a half-move of both legs, one block per leg: append each live game's move at ply `half`, check that the other
// model's tree took the previous move (other_status, from the second half-move on), tally and record the games that ended
// (BlackWin for the side that opened: the network in leg 0), and compact the leg's live list stably -- both models' tree ids
// and the moves, which the other model's trees take next -- so a game's two trees stay in step.  Block 0 also copies the device
// error word next to the live counts.
__global__ void __launch_bounds__(kAdvanceThreads) k_match_advance(int pairs, int first_tree, int half, int live0, int live1, int32_t *ids,
                                                                   int32_t *actions, const int8_t *status, const int8_t *other_status,
                                                                   int8_t *moves, int8_t *final_status, int32_t *counters,
                                                                   uint32_t *dev_error) {
    __shared__ int warp_kept[kAdvanceThreads / 32];
    __shared__ int kept_before;
    const int leg = blockIdx.x, n = leg ? live1 : live0;
    int32_t *ids_net = ids + leg * pairs, *ids_opp = ids + (2 + leg) * pairs, *act = actions + leg * pairs;
    const int8_t *st_leg = status + leg * pairs, *ost_leg = other_status + leg * pairs;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) kept_before = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += kAdvanceThreads) {
        const int i = c0 + threadIdx.x;
        bool keep = false;
        int32_t tn = 0, to = 0, a = 0;
        if (i < n) {
            tn = ids_net[i];
            to = ids_opp[i];
            a = act[i];
            const int g = tn - first_tree;
            const int st = st_leg[i];
            moves[(size_t)g * kCells + half] = (int8_t)a;
            if (half > 0 && ost_leg[i] != kInProgress) atomicOr(dev_error, 16u);
            if (st == kInProgress) {
                keep = true;
            } else if (st == kDraw || st == kBlackWin || st == kWhiteWin) {
                final_status[g] = (int8_t)st;
                const int opener = g < pairs ? 0 : 1;
                atomicAdd(&counters[st == kDraw ? 2 : (st == kBlackWin ? opener : 1 - opener)], 1);
            } else {
                atomicOr(dev_error, 16u);  // Option::None: the move was refused -- the game could never end
            }
        }
        const uint32_t b = __ballot_sync(kFullMask, keep);
        if (lane == 0) warp_kept[warp] = __popc(b);
        __syncthreads();  // every entry of this chunk has been read before any is overwritten
        int dst = kept_before + __popc(b & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) dst += warp_kept[w];
        if (keep) {
            ids_net[dst] = tn;
            ids_opp[dst] = to;
            act[dst] = a;
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < kAdvanceThreads / 32; ++w) kept_before += warp_kept[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counters[4 + leg] = kept_before;
        if (leg == 0) counters[3] = (int32_t)atomicOr(dev_error, 0u);  // read back with the live counts
    }
}

// ---- the tournament (omk_tournament): omk_match's bookkeeping over n participants and their n(n-1)/2 pairings ----
// With t.naive, participant 0 is the naive player: it has no trees (its side of its pairings is reserved and never touched),
// and it moves by k_naive_move on the roots of its opponents' trees, which hold the current positions.
// pairing p = (a, b), a < b, in lexicographic order
__device__ __forceinline__ void tourney_pairing(int p, int n, int &a, int &b) {
    a = 0;
    while (p >= n - 1 - a) p -= n - 1 - a++;
    b = a + 1 + p;
}
// the r-th pairing (in pairing order) of model m, and m's side in it (0 left, 1 right)
__device__ __forceinline__ void tourney_model_pairing(int m, int r, int n, int &p, int &side) {
    const int a = r < m ? r : m, b = r < m ? m : r + 1;
    p = a * n - a * (a + 1) / 2 + (b - a - 1);
    side = r < m ? 1 : 0;
}

// A fresh tournament: pairing p's trees are first_tree + 4 * pairs * p + omk_match's layout, every game live, nothing tallied.
// Model m's list gids[m] holds every tree of m (both legs of each of its pairings, in pairing order) with the tree's stream in
// gstr[m], for Agent::new under m's weights.
__global__ void k_tourney_init(TourneyState t) {
    const int Q = t.pairs, P = t.n * (t.n - 1) / 2, per_model = (t.n - 1) * 2 * Q;
    const long long total = (long long)P * 2 * Q * kCells;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        t.moves[k] = -1;
        if (k < 4LL * Q * P) t.ids[k] = t.first_tree + (int)k;
        if (k < 2LL * Q * P) {
            t.actions[k] = -1;
            t.final_status[k] = kInProgress;
        }
        if (k < 2 * P) t.live[k] = Q;
        if (k < 3 * P) t.counters[k] = 0;
        if (k < (long long)t.n * per_model) {
            const int m = (int)(k / per_model), i = (int)(k % per_model), w = i % (2 * Q);
            int p, side;
            tourney_model_pairing(m, i / (2 * Q), t.n, p, side);
            t.gids[(size_t)m * t.gcap + i] = t.first_tree + 4 * Q * p + side * 2 * Q + w;
            t.gstr[(size_t)m * t.gcap + i] = (uint32_t)(w % Q);
        }
    }
}

// After half-move `half`, one block per (pairing, leg): k_match_advance for that leg, with the movers' actions and statuses
// read out of their model's group segment.  The left model moves in leg half % 2, the right one in the other leg.  The naive
// player's statuses are those of its moves on the board (k_naive_move); it has no tree to take the other side's move, so
// there is no other_status to check.
__global__ void __launch_bounds__(kAdvanceThreads) k_tourney_advance(TourneyState t, int half, uint32_t *dev_error) {
    __shared__ int warp_kept[kAdvanceThreads / 32];
    __shared__ int kept_before;
    const int p = blockIdx.x >> 1, leg = blockIdx.x & 1, Q = t.pairs;
    int a_model, b_model;
    tourney_pairing(p, t.n, a_model, b_model);
    const int mover = leg == half % 2 ? a_model : b_model;
    const bool check_other = half > 0 && !(t.naive && mover == 0);
    const int n = t.live[2 * p + leg];
    const size_t seg = (size_t)mover * t.gcap + t.off[2 * p + leg];
    const int32_t *g_act = t.gact + seg;
    const int8_t *g_st = t.gst + seg, *g_ost = t.gost + seg;
    int32_t *ids_l = t.ids + (size_t)(4 * p + leg) * Q, *ids_r = t.ids + (size_t)(4 * p + 2 + leg) * Q;
    int32_t *act = t.actions + (size_t)(2 * p + leg) * Q;
    const int base = t.first_tree + 4 * Q * p;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) kept_before = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += kAdvanceThreads) {
        const int i = c0 + threadIdx.x;
        bool keep = false;
        int32_t tl = 0, tr = 0, a = 0;
        if (i < n) {
            tl = ids_l[i];
            tr = ids_r[i];
            a = g_act[i];
            const int g = tl - base;
            const int st = g_st[i];
            const size_t row = (size_t)p * 2 * Q + g;
            t.moves[row * kCells + half] = (int8_t)a;
            if (check_other && g_ost[i] != kInProgress) atomicOr(dev_error, 16u);
            if (st == kInProgress) {
                keep = true;
            } else if (st == kDraw || st == kBlackWin || st == kWhiteWin) {
                t.final_status[row] = (int8_t)st;
                const int opener = g < Q ? 0 : 1;
                atomicAdd(&t.counters[3 * p + (st == kDraw ? 2 : (st == kBlackWin ? opener : 1 - opener))], 1);
            } else {
                atomicOr(dev_error, 16u);  // Option::None: the move was refused -- the game could never end
            }
        }
        const uint32_t b = __ballot_sync(kFullMask, keep);
        if (lane == 0) warp_kept[warp] = __popc(b);
        __syncthreads();  // every entry of this chunk has been read before any is overwritten
        int dst = kept_before + __popc(b & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) dst += warp_kept[w];
        if (keep) {
            ids_l[dst] = tl;
            ids_r[dst] = tr;
            act[dst] = a;
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < kAdvanceThreads / 32; ++w) kept_before += warp_kept[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) t.live[2 * p + leg] = kept_before;
}

// The groups of half-move `half`, one block per model m: the concatenation, in pairing order, of the live lists of the legs
// m moves in (its trees, and the moves they take first: the other side's previous ones), each segment's offset, and the
// group's size.  The naive player's group lists its opponents' trees of those legs: the boards it reads.  Block 0 also
// copies the device error word next to the sizes.
__global__ void k_tourney_gather(TourneyState t, int half, uint32_t *dev_error) {
    const int m = blockIdx.x, Q = t.pairs;
    int32_t *g_ids = t.gids + (size_t)m * t.gcap, *g_act = t.gact + (size_t)m * t.gcap;
    int o = 0;
    for (int r = 0; r < t.n - 1; ++r) {
        int p, side;
        tourney_model_pairing(m, r, t.n, p, side);
        const int leg = (half + side) % 2, cnt = t.live[2 * p + leg], trees = t.naive && m == 0 ? 1 - side : side;
        const int32_t *src_ids = t.ids + (size_t)(4 * p + 2 * trees + leg) * Q, *src_act = t.actions + (size_t)(2 * p + leg) * Q;
        for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
            g_ids[o + j] = src_ids[j];
            g_act[o + j] = src_act[j];
        }
        if (threadIdx.x == 0) t.off[2 * p + leg] = o;
        o += cnt;
    }
    if (threadIdx.x == 0) {
        t.back[1 + m] = o;
        if (m == 0) t.back[0] = (int32_t)atomicOr(dev_error, 0u);  // read back with the sizes
    }
}

// ---- launchers ----
static NaiveArgs naive_args(int n, uint64_t key, int32_t *actions, uint8_t *forced) {
    NaiveArgs a{};
    a.n = n;
    a.key = key;
    a.actions = actions;
    a.forced = forced;
    return a;
}
void launch_naive_move_boards(omk_ctx *c, const uint8_t *boards, const uint8_t *turns, const uint32_t *streams, int n, uint64_t key,
                              int32_t *actions, uint8_t *forced) {
    if (n <= 0) return;
    NaiveArgs a = naive_args(n, key, actions, forced);
    a.boards = boards;
    a.turns = turns;
    a.streams = streams;
    k_naive_move<<<(n + kNaiveWarps - 1) / kNaiveWarps, kNaiveWarps * 32, 0, c->stream>>>(a);
    c->launches++;
}
void launch_naive_move_trees(omk_ctx *c, const int32_t *ids, int n, int first_tree, const int32_t *ply, uint64_t key, int32_t *actions) {
    if (n <= 0) return;
    NaiveArgs a = naive_args(n, key, actions, nullptr);
    a.ids = ids;
    a.nodes = c->tree_nodes;
    a.cap_nodes = c->cap_nodes;
    a.first_tree = first_tree;
    a.ply = ply;
    k_naive_move<<<(n + kNaiveWarps - 1) / kNaiveWarps, kNaiveWarps * 32, 0, c->stream>>>(a);
    c->launches++;
}
void launch_tourney_naive_move(omk_ctx *c, const TourneyState &t, int half, int n, uint64_t key) {
    if (n <= 0) return;
    NaiveArgs a = naive_args(n, key, t.gact, nullptr);
    a.ids = t.gids;
    a.nodes = c->tree_nodes;
    a.cap_nodes = c->cap_nodes;
    a.first_tree = t.first_tree;
    a.pairs = t.pairs;
    a.half = half;
    a.status = t.gst;
    k_naive_move<<<(n + kNaiveWarps - 1) / kNaiveWarps, kNaiveWarps * 32, 0, c->stream>>>(a);
    c->launches++;
}
void launch_eval_init(omk_ctx *c, int episodes, int first_tree, int32_t *ids, int32_t *ply, int8_t *moves, int8_t *final_status,
                      int32_t *counters) {
    const int total = episodes * kCells;
    k_eval_init<<<(total + 255) / 256, 256, 0, c->stream>>>(episodes, first_tree, ids, ply, moves, final_status, counters);
    c->launches++;
}
void launch_eval_advance(omk_ctx *c, int32_t *ids, int n, const int32_t *actions, const int8_t *status, int first_tree, int32_t *ply,
                         int8_t *moves, int8_t *final_status, int32_t *counters) {
    k_eval_advance<<<1, kAdvanceThreads, 0, c->stream>>>(ids, n, actions, status, first_tree, ply, moves, final_status, counters,
                                                          c->dev_error);
    c->launches++;
}
void launch_match_init(omk_ctx *c, int pairs, int first_tree, int32_t *ids, uint32_t *streams, int8_t *moves, int8_t *final_status,
                       int32_t *counters) {
    const int total = 2 * pairs * kCells;
    k_match_init<<<(total + 255) / 256, 256, 0, c->stream>>>(pairs, first_tree, ids, streams, moves, final_status, counters);
    c->launches++;
}
void launch_match_advance(omk_ctx *c, int pairs, int first_tree, int half, const int *live, int32_t *ids, int32_t *actions,
                          const int8_t *status, const int8_t *other_status, int8_t *moves, int8_t *final_status, int32_t *counters) {
    k_match_advance<<<2, kAdvanceThreads, 0, c->stream>>>(pairs, first_tree, half, live[0], live[1], ids, actions, status, other_status,
                                                           moves, final_status, counters, c->dev_error);
    c->launches++;
}
void launch_tourney_init(omk_ctx *c, const TourneyState &t) {
    const long long total = (long long)t.n * (t.n - 1) / 2 * 2 * t.pairs * kCells;
    const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    k_tourney_init<<<blocks, 256, 0, c->stream>>>(t);
    c->launches++;
}
void launch_tourney_advance(omk_ctx *c, const TourneyState &t, int half) {
    k_tourney_advance<<<t.n * (t.n - 1), kAdvanceThreads, 0, c->stream>>>(t, half, c->dev_error);
    c->launches++;
}
void launch_tourney_gather(omk_ctx *c, const TourneyState &t, int half) {
    k_tourney_gather<<<t.n, 256, 0, c->stream>>>(t, half, c->dev_error);
    c->launches++;
}

}  // namespace omk
