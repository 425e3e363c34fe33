// omk_internal.h -- host-side context and kernel launcher prototypes (not part of the ABI).
#pragma once
#include <cstdint>
#include <memory>
#include <utility>
#include <vector>
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "../../include/omok_b200.h"
#include "omk_device.cuh"

namespace omk {

constexpr int kMaxBatchPerTree = 64;  // per-tree requests per round (evaluate_batch_size)
constexpr int kNetTensors = 31;
constexpr int kModelSlots = 16;  // weight sets per context: 0 the network, 1 the opponent, 2 .. 15 further models (omk_model_*)

enum ApplyMode { kApplySearch = 0, kApplyNewGame = 1, kApplyEnsure = 2 };

// Owner of one allocation of `count` T: device memory (DeviceMem), or pinned host memory (PinnedMem).  Move-only, released on
// destruction; converts to the raw pointer, so kernels and launchers take T * unchanged.
struct DeviceMem {
    static cudaError_t alloc(void **p, size_t bytes) { return cudaMalloc(p, bytes); }
    static void release(void *p) { cudaFree(p); }
};
struct PinnedMem {
    static cudaError_t alloc(void **p, size_t bytes) { return cudaHostAlloc(p, bytes, cudaHostAllocDefault); }
    static void release(void *p) { cudaFreeHost(p); }
};
template <typename T, typename Mem = DeviceMem>
class Buf {
  public:
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    Buf(Buf &&o) noexcept : p_(std::exchange(o.p_, nullptr)), count_(std::exchange(o.count_, 0)) {}
    Buf &operator=(Buf &&o) noexcept {
        if (this != &o) {
            reset();
            p_ = std::exchange(o.p_, nullptr);
            count_ = std::exchange(o.count_, 0);
        }
        return *this;
    }
    ~Buf() { reset(); }
    operator T *() const { return p_; }
    T *get() const { return p_; }
    size_t bytes() const { return sizeof(T) * count_; }
    void reset() {
        if (p_) Mem::release(p_);
        p_ = nullptr;
        count_ = 0;
    }
    // release the current allocation, then allocate `count` elements (on failure the handle is left empty)
    cudaError_t alloc(size_t count) {
        reset();
        void *p = nullptr;
        const cudaError_t e = Mem::alloc(&p, sizeof(T) * count);
        if (e != cudaSuccess) return e;
        p_ = static_cast<T *>(p);
        count_ = count;
        return cudaSuccess;
    }
    // grow-only: a request beyond the capacity synchronises `s` (work queued there may still use the old allocation), then
    // allocates `count` rounded up to a multiple of `round` elements
    cudaError_t grow(cudaStream_t s, size_t count, size_t round = 1) {
        if (count <= count_) return cudaSuccess;
        const cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return e;
        return alloc((count + round - 1) / round * round);
    }

  private:
    T *p_ = nullptr;
    size_t count_ = 0;
};
template <typename T>
using PinnedBuf = Buf<T, PinnedMem>;

// Each group below is allocated into a local instance and moved into its owner only when every allocation succeeded, so no
// call can find half a group.
struct FcImages {  // fp16-split tensor-core path (fc_f16.cu): weights scaled by a power of two, then split hi/lo
    Buf<__half> fc0_wt_h16, fc0_wt_l16;    // [512][10368] K-major
    Buf<__half> fc1_wt_h16, fc1_wt_l16;    // [512][512]
    Buf<__half> heads_wt_h16, heads_wt_l16;  // [128][512]: rows 0..80 policy, 81 value, rest 0
    Buf<float> fc_inv_scale;               // [3] 2^-s of fc0, fc1, heads
    Buf<uint32_t> fc_absmax;               // [3] max |w| bits
};
struct TowerImages {  // tower_f16.cu
    Buf<uint8_t> tower16_wimg;       // 3 x 36 KB pre-swizzled B-operand images
    Buf<float> tower16_pimg;         // fp32 stem / bias / depthwise parameters + inverse scales
    Buf<uint32_t> tower16_absmax;    // [9]
};
struct WeightMaps {  // tensor maps (fc_f16.cu) over one model's fp16 weight images
    CUtensorMap map0_b_hi, map0_b_lo;    // fc0 (B boxes of 128 rows: the pair kernel loads half tiles)
    CUtensorMap map0s_b_hi, map0s_b_lo;  // fc0 weights with 256-row boxes (one-CTA split-K kernel for small batches)
    CUtensorMap map1_b_hi, map1_b_lo;    // fc1 (B boxes of 256 rows)
    CUtensorMap map2_b_hi, map2_b_lo;    // heads (B = all 128 padded output rows)
    bool weights_ready = false;
};
// Everything derived from one set of weights.  The context holds kModelSlots: the network (slot 0, `net`: every entry point,
// the trainer), the opponent (slot 1, `opp`: omk_opponent_eval, omk_match) and further models (slots 2 .., `more`:
// omk_model_eval, omk_tournament).  The evaluator reads the active one, omk_ctx::model.
struct NetWeights : FcImages, TowerImages, WeightMaps {
    Buf<float> t[kNetTensors];  // device copies in checkpoint order
    Buf<float> heads_w;         // [512][128]: cols 0..80 policy, col 81 value, rest 0
    Buf<float> heads_b;         // [128]
    std::vector<uint8_t> tower16_params_host;  // host copy of the tower's fp32 parameter image (kernel argument of k_tower16)
    bool loaded = false;
};

struct ActMaps {  // tensor maps (fc_f16.cu) over one workspace's fp16 activation buffers
    CUtensorMap map0_a_hi, map0_a_lo, map1_a_hi, map1_a_lo, map2_a_hi, map2_a_lo;
    CUtensorMap tower_st_hi, tower_st_lo;  // k_tower16's write-out into act0
};
struct Activations {  // activation buffers [act_rows] of the network, allocated on first use (ensure_activations)
    int act_rows = 0;
    bool act_fp32 = false;            // the fp32 buffers of the CUDA-core A/B kernels exist (act0, act1)
    Buf<__half> act0_h16, act0_l16;   // [act_rows][10368] fp16 hi/lo split of the tower output == fc0's A operand
    Buf<__half> act1_h16, act1_l16;   // [act_rows][512] fp16 hi/lo split of fc0's output == fc1's A operand
    Buf<__half> act2_h16, act2_l16;   // [act_rows][512] fp16 hi/lo split of fc1's output == the heads' A operand
    Buf<float> act2;                  // [act_rows][512] fc1 output (fp32: CUDA-core heads, debugging)
    Buf<float> logits;                // [act_rows][128]
    Buf<float> act0;                  // [act_rows][10368] fp32 tower output (CUDA-core A/B kernels only)
    Buf<float> act1;                  // [act_rows][512]   fp32 fc0 output   (CUDA-core A/B kernels only)
    ActMaps maps;                     // encoded with the buffers (fc16_encode_act_maps)
};
// One search lane's evaluator buffers (LaneScope in omk_api.cu swaps the whole workspace): request/response buffers
// [max_rows], the activations, and the lane's fc0 scratch
struct Workspace : Activations {
    int max_rows = 0;
    Buf<NNIn> nn_in;            // [max_rows]
    Buf<uint32_t> req_tree;     // [max_rows]
    Buf<uint32_t> req_node;     // [max_rows]
    Buf<float> P;               // [max_rows][96]
    Buf<float> V;               // [max_rows]
    Buf<uint32_t> n_req;        // device counter
    Buf<uint32_t> slot_base, slot_count;  // [capacity_trees]
    Buf<int32_t> ids;           // [capacity_trees] device copy of the call's id list
    Buf<int32_t> actions;       // [capacity_trees]
    Buf<uint8_t> modes;         // [capacity_trees]
    Buf<float> temps;           // [capacity_trees]
    Buf<int8_t> status;         // [capacity_trees]
    Buf<float> policy_out;      // [capacity_trees][81]
    Buf<uint32_t> streams;      // [capacity_trees]
    Buf<float> splitk_partial;  // [chunks][rows][512] fp32 partial sums of the split-K fc0 (grow-only)
    Buf<float4> bal_partial;    // tail-balancing scratch of the pair fc0: [units][F_BAL_UNIT_F4] (grow-only)
    Buf<uint32_t> bal_flags;    // [256]
};

// Replay memory on the device (replay_kernels.cu; DESIGN.md 2).  Row a (absolute: rows added since the last reset) lives
// at a % cap; logical row i (0 = oldest) is absolute row added - len + i.
struct ReplayRing {  // kernel argument: a view of ReplayStore
    uint8_t *boards;  // [cap][81]
    uint8_t *turns;   // [cap]
    float *pi;        // [cap][81]
    float *z;         // [cap]
    long long cap;
};
struct ReplayStore {
    Buf<uint8_t> boards, turns;
    Buf<float> pi, z;
    long long cap = 0;
    ReplayRing view() const { return {boards, turns, pi, z, cap}; }
};
struct ReplayCounters {  // device; advanced by the per-ply commit
    long long added, len, episodes;
    uint32_t done, pad;  // arrival counter of the commit's blocks (re-armed)
};
struct ReplayStaging {  // the driver's unfinished games: [games][81 plies][81] boards and policies, [games] ply counts
    int games = 0;      // 0: the driver does not feed the replay
    Buf<uint8_t> boards;
    Buf<float> pi;
    Buf<int32_t> len;
};
struct Replay {
    ReplayStore ring;
    Buf<ReplayCounters> counters;
    long long added = 0, len = 0, episodes = 0;  // host copy of *counters, refreshed by omk_selfplay_run
    ReplayStaging stage;
    cudaStream_t stream = nullptr;      // the per-ply commits
    cudaEvent_t ev_commit = nullptr;    // the last commit enqueued
};

// opaque to this header; their deleters live with them
struct Fc16State;
struct TrainState;
struct Fc16StateFree { void operator()(Fc16State *s) const; };   // fc_f16.cu
struct TrainStateFree { void operator()(TrainState *t) const; };  // train_kernels.cu

}  // namespace omk

struct omk_prof_span {
    cudaEvent_t a, b;
    int kind;
};

struct omk_ctx {
    ~omk_ctx();  // synchronises every stream of the context before any buffer is released (omk_api.cu)
    int device = 0;
    // profiling spans (CUDA events on the context stream); level 0 none, 1 fc0 only, 2 all families
    int prof_level = 0;
    std::vector<omk_prof_span> prof_spans;
    std::vector<cudaEvent_t> prof_pool;
    int n_sms = 0;
    int cap_envs = 0, cap_trees = 0, cap_nodes = 0;
    uint64_t seed = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    int64_t h2d_bytes = 0, d2h_bytes = 0;  // host <-> device bytes copied by the API layer since creation
    // Second search lane: large searches split their trees into two halves that run as two independent chains of
    // kernels on two streams with two evaluator workspaces.  Trees never interact, so the split changes no result; the
    // latency-bound tree kernels of one half then overlap the (tensor-bound, register-light) fc0 of the other half.
    // `stream` / `ws` above are the lane in use: LaneScope (omk_api.cu) swaps them with these for lane 1.
    cudaStream_t lane1_stream = nullptr;
    omk::Workspace lane1_ws;
    cudaEvent_t lane_fork = nullptr, lane_join = nullptr;
    int lane_min_trees = 768;       // searches over fewer trees stay on one lane: each lane should still fill an fc0 wave (env OMK_LANE_MIN_TREES; 0 disables lanes)
    // grow-only device scratch of the granular host-buffer calls (env_step, env_get, net_eval, ...): no cudaMalloc /
    // cudaFree (an implicit device synchronisation each) per call, nothing to leak on an error return
    omk::Buf<uint8_t> scratch[3];
    std::vector<uint8_t> id_seen;   // host scratch of stage_ids: duplicate detection over an id list
    int id_base = 0;                // first tree id of the lane in use when the id list is the identity

    omk::Buf<omk::EnvRec> envs;
    omk::Buf<omk::TreeHdr> tree_hdrs;
    omk::Buf<uint8_t> tree_nodes;    // [cap_trees][cap_nodes][kNodeBytes]
    omk::Buf<uint16_t> remap;        // [cap_trees][cap_nodes] compaction scratch
    omk::Buf<uint32_t> dev_error;    // sticky device error word
    omk::Buf<unsigned long long> dev_sims;  // simulations counter

    omk::NetWeights net;            // the network
    omk::NetWeights opp;            // the opponent, slot 1 (omk_opponent_load_params / omk_opponent_from_net); buffers allocated on first load
    omk::NetWeights more[omk::kModelSlots - 2];  // slots 2 .. (omk_model_load_params / omk_model_from_net); buffers allocated on first load
    omk::NetWeights *model = &net;  // the weights the evaluator reads: `net`, or another slot inside a ModelScope (omk_api.cu)
    omk::NetWeights &slot(int s) { return s == 0 ? net : (s == 1 ? opp : more[s - 2]); }
    omk::Workspace ws;
    int virtual_loss = 0;           // opt-in, non-reference search mode (omk_search_set_virtual_loss); refused with the parity evaluator
    int fc0_balance = 0;            // fc0 tail balancing of the CTA-pair kernel (fc_f16.cu FcBal): 0 off (default), 1 on
    int fc0_chunk = 9;              // k-blocks of fc0 accumulated in tensor memory per drain: 9 (default) or 3 (finer, more accurate; fc_f16.cu)
    int fc0_mode = 1;               // fc0 + fc1: 1 = tcgen05 3xFP16 k_fc16 (the product path), 0 = fp32 CUDA-core k_gemm (A/B check only)
    std::unique_ptr<omk::Fc16State, omk::Fc16StateFree> fc16_state;  // the device's occupancy answers for the fp16-split path (fc_f16.cu)
    int tower16_pairs = 0;          // resident CTA pairs of k_tower16 (0 = not queried yet)
    std::unique_ptr<omk::TrainState, omk::TrainStateFree> train_state;  // trainer step workspace, Adadelta slots, optional NCCL communicator (train_kernels.cu)
    int train_n = 0;                // positions of the minibatch currently on the device (omk_train_backward)
    bool net_pack_dirty = false;    // omk_train_apply changed the fp32 weights: the tensor-core operand images (and a running self-play
                                    // driver's cached root prior) are rebuilt before the next network evaluation (ensure_packed in omk_api.cu)
    int tower_mode = 1;             // tower: 1 = tcgen05 3xFP16 k_tower16 (the product path), 0 = fp32 CUDA-core k_tower (A/B check only)

    // self-play driver state
    omk_selfplay_config sp_cfg{};
    bool sp_active = false;
    omk::Buf<int32_t> sp_ply;         // [n_games] device ply counters
    omk::Buf<uint8_t> sp_buf;         // per-game scratch (ids, actions, modes, status, cached root policy)
    // Transition ring of the self-play driver (BASELINE config 4: positions streamed to the host replay buffer): kSpRing
    // ply slots on the device, mirrored in pinned host memory; a ply's slice leaves on `sp_copy_stream` while the next
    // plies search.  Allocated by omk_selfplay_begin for sp_cfg.n_games.
    static constexpr int kSpRing = 4;
    omk::Buf<uint8_t> sp_ring_dev;    // kSpRing x [boards n*81 | policy n*81 f32 | actions n i32 | status n]
    omk::PinnedBuf<uint8_t> sp_ring_host;
    size_t sp_ring_slot_bytes = 0;
    cudaStream_t sp_copy_stream = nullptr;
    cudaEvent_t sp_ev_rec[kSpRing][2] = {}, sp_ev_copy[kSpRing] = {};
    omk::Replay rp;                   // device replay memory (omk_replay_reset); fed by the driver when it exists at omk_selfplay_begin
    omk::Buf<uint8_t> eval_buf;       // omk_eval_naive's, omk_match's and omk_tournament's per-call state (grow-only)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

namespace omk {

// ---- launchers (each increments ctx->launches) ----
// env_kernels.cu
void launch_env_reset(omk_ctx *c, const int32_t *ids_dev, int n);
void launch_env_step(omk_ctx *c, const int32_t *ids_dev, const uint8_t *actions_dev, int n, int8_t *status_dev,
                     uint32_t *legal_dev);
void launch_env_get(omk_ctx *c, const int32_t *ids_dev, int n, uint8_t *boards_dev, uint8_t *turns_dev,
                    uint16_t *legal_dev);
void launch_env_set(omk_ctx *c, const int32_t *ids_dev, int n, const uint8_t *boards_dev, const uint8_t *turns_dev);
void launch_env_encode(omk_ctx *c, const int32_t *ids_dev, int n, int mode, float *out_dev);
void launch_env_playout(omk_ctx *c, int n, int plies, uint8_t *actions_dev, int8_t *status_dev);
void launch_pack_boards(omk_ctx *c, const uint8_t *boards_dev, const uint8_t *turns_dev, int n, int mode);

// tree_kernels.cu
// only_if_terminal != nullptr: restart only slots whose status is terminal, keep their random stream running;
// root_policy != nullptr: install that raw policy instead of queueing an evaluation
void launch_new_games(omk_ctx *c, const int32_t *ids_dev, int n, const uint32_t *streams_dev,
                      const int8_t *only_if_terminal, const float *root_policy);
void launch_root_noise(omk_ctx *c, const int32_t *ids_dev, int n, float epsilon, float alpha);
void launch_select_expand(omk_ctx *c, const int32_t *ids_dev, int n, int batch);
void launch_apply(omk_ctx *c, const int32_t *ids_dev, int n, int mode);
void launch_sample(omk_ctx *c, const int32_t *ids_dev, int n, const uint8_t *modes_dev, const float *temps_dev,
                   int32_t *actions_dev, float *policy_dev, uint8_t *valid_dev);
void launch_ensure_prepare(omk_ctx *c, const int32_t *ids_dev, const int32_t *actions_dev, int n);
void launch_play(omk_ctx *c, const int32_t *ids_dev, const int32_t *actions_dev, int n, int8_t *status_dev);
void launch_root_children(omk_ctx *c, int tree, int32_t *actions_dev, unsigned long long *n_dev, float *w_dev,
                          float *p_dev, int32_t *len_dev, float *policy_dev, uint32_t *misc_dev);
void launch_eval_hash(omk_ctx *c, int rows_bound);
void launch_pool_get_envs(omk_ctx *c, const int32_t *ids_dev, int n, uint8_t *boards_dev, uint8_t *turns_dev,
                          uint16_t *legal_dev, int8_t *status_dev);
void launch_reset_requests(omk_ctx *c);
void launch_sp_prepare(omk_ctx *c, int g0, int n, int32_t *mover, int32_t *other, uint8_t *modes, float *temps);
void launch_sp_record(omk_ctx *c, int n, const int32_t *mover, const int32_t *actions, const float *policy_in,
                      uint8_t *boards_out, float *policy_out, int32_t *actions_out);
void launch_sp_advance(omk_ctx *c, int g0, int n, const int8_t *status, unsigned long long *counters);

// replay_kernels.cu: stage a lane's recorded ply (ring-slot boards / policies of games g0..g0+n-1) on c->stream; commit the
// ply's finished episodes on the replay stream; sample `steps` minibatches of m logical rows; gather + encode one minibatch;
// copy rows out for omk_replay_get
void launch_rp_stage(omk_ctx *c, int g0, int n, const uint8_t *boards, const float *policy);
void launch_rp_commit(omk_ctx *c, int n, const int8_t *status);
void launch_rp_sample(omk_ctx *c, uint64_t seed, long long first_step, int steps, long long len, int m, int64_t *rows);
void launch_rp_gather(omk_ctx *c, const int64_t *rows, int m, float *img, float *pi, float *z);
void launch_rp_get(omk_ctx *c, const int64_t *rows, int n, uint8_t *boards, uint8_t *turns, float *pi, float *z);

// eval_kernels.cu: the naive player's move (trainer.rs:506-537) for positions given as cells + turns, or for the roots of
// the live trees of omk_eval_naive; that driver's set-up and its bookkeeping after each half-move (move records, tallies,
// stable compaction of the live list; counters = {BlackWin, WhiteWin, Draw, live})
void launch_naive_move_boards(omk_ctx *c, const uint8_t *boards, const uint8_t *turns, const uint32_t *streams, int n, uint64_t key,
                              int32_t *actions, uint8_t *forced);
void launch_naive_move_trees(omk_ctx *c, const int32_t *ids, int n, int first_tree, const int32_t *ply, uint64_t key, int32_t *actions);
void launch_eval_init(omk_ctx *c, int episodes, int first_tree, int32_t *ids, int32_t *ply, int8_t *moves, int8_t *final_status,
                      int32_t *counters);
void launch_eval_advance(omk_ctx *c, int32_t *ids, int n, const int32_t *actions, const int8_t *status, int first_tree, int32_t *ply,
                         int8_t *moves, int8_t *final_status, int32_t *counters);
// omk_match (DESIGN.md 4): its set-up, and its bookkeeping after each half-move of both legs.  ids = [model][leg][pairs] tree
// ids of the live games (network 0, opponent 1), actions / status / other_status = [leg][pairs], counters = {network wins,
// opponent wins, draws, device error word, live in leg 0, live in leg 1}
void launch_match_init(omk_ctx *c, int pairs, int first_tree, int32_t *ids, uint32_t *streams, int8_t *moves, int8_t *final_status,
                       int32_t *counters);
void launch_match_advance(omk_ctx *c, int pairs, int first_tree, int half, const int *live, int32_t *ids, int32_t *actions,
                          const int8_t *status, const int8_t *other_status, int8_t *moves, int8_t *final_status, int32_t *counters);
// omk_tournament (DESIGN.md 4): n participants, P = n(n-1)/2 pairings (i < j, lexicographic), `pairs` games per leg of each.
// naive: participant 0 is the naive player (omk_tournament_naive), the others are models; otherwise all n are models.  The
// per-pairing state is omk_match's: ids [P][side][leg][pairs] (left 0, right 1), actions [P][leg][pairs], live [P][leg],
// counters [P][3] = {left wins, right wins, draws}, moves [P][2 * pairs][81], final status [P][2 * pairs].  Model m's group
// (its movers of one half-move, over all its pairings in order) is [m][gcap] in gids / gact / gst / gost, and off [P][leg] is
// where a (pairing, leg)'s movers sit in their model's group.  back = {device error word, group size of each model}.
struct TourneyState {
    int n, pairs, first_tree, gcap, naive;
    int32_t *ids, *actions, *live, *off, *counters, *back;
    int32_t *gids, *gact;  // [n][gcap]
    int8_t *gst, *gost;    // [n][gcap]: the movers' play_action statuses, and their trees' statuses taking the other side's move
    uint32_t *gstr;        // [n][gcap]: random streams of k_tourney_init's per-model lists of all the model's trees
    int8_t *moves, *final_status;
};
// set-up: every pairing's trees, all games live, nothing tallied; gids / gstr = every tree of each model with its stream
void launch_tourney_init(omk_ctx *c, const TourneyState &t);
// after half-move `half`: record, check, tally and compact each (pairing, leg) from its movers' group segment
void launch_tourney_advance(omk_ctx *c, const TourneyState &t, int half);
// the groups of half-move `half` from the compacted lists: gids, gact (the move each tree takes in stage 0), off, back
void launch_tourney_gather(omk_ctx *c, const TourneyState &t, int half);
// the naive player's half-move `half`: its n moves, and their statuses on the board, from the roots of the trees of its group
// (participant 0's gids) into its gact / gst; key = mix64(seed ^ kNaiveKey)
void launch_tourney_naive_move(omk_ctx *c, const TourneyState &t, int half, int n, uint64_t key);

// omk_api.cu: open / close a profiling span of kernel family `kind` (no-op below min_level)
bool prof_begin(omk_ctx *c, int kind, int min_level);
void prof_end(omk_ctx *c, bool opened);

// net_kernels.cu
bool net_forward(omk_ctx *c, const float *images_dev /* or nullptr: use ws.nn_in */, int max_rows);  // false: nothing usable in ws.P / ws.V
void net_pack_heads(omk_ctx *c);
void launch_net_init_random(omk_ctx *c, uint64_t seed);

// omk_api.cu: size the activation buffers for `rows` evaluator rows (fp32 A/B buffers only when a CUDA-core mode is on)
bool ensure_activations(omk_ctx *c, int rows);

// fc_f16.cu
bool fc16_prepare_weights(omk_ctx *c);
bool launch_fc0_f16(omk_ctx *c, int rows_bound);
bool launch_fc1_f16(omk_ctx *c, int rows_bound);
bool launch_heads_f16(omk_ctx *c, int rows_bound);
// encode a.maps over a's fp16 buffers (ensure_activations, whenever it (re)allocates them)
bool fc16_encode_act_maps(Activations &a);
void launch_f32_to_split16(omk_ctx *c, const float *x, __half *hi, __half *lo, long long n);
void launch_split16_to_f32(omk_ctx *c, const __half *hi, const __half *lo, float *x, long long n);

// train_kernels.cu: every function returns nullptr on success or a message
const char *train_backward_step(omk_ctx *c, const float *images, const float *pi, const float *z, int n, float **grads_dev);
const char *train_apply_step(omk_ctx *c);
const char *train_report_losses(omk_ctx *c, int n, float *out3);
// the replay path: the minibatch buffers for n positions (filled on the device), then the same forward / losses / backward,
// and the reporting forward with its losses left in device memory (dst3)
const char *train_minibatch_buffers(omk_ctx *c, int n, float **img, float **pi, float **z);
const char *train_backward_resident(omk_ctx *c, int n);
const char *train_report_losses_device(omk_ctx *c, int n, float *dst3);
float *train_grad_buffer(omk_ctx *c);
void train_reset_optimizer(omk_ctx *c);
const char *train_comm_unique_id(omk_ctx *c, uint8_t *out128);
const char *train_comm_init(omk_ctx *c, const uint8_t *id128, int nranks, int rank);
const char *train_comm_destroy(omk_ctx *c);

// tower_f16.cu
bool tower16_prepare_weights(omk_ctx *c);
bool launch_tower_f16(omk_ctx *c, const float *images_dev, int rows_bound);
void tower16_read_timing(long long *out64);

}  // namespace omk
