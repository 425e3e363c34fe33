// omk_internal.h -- host-side context and kernel launcher prototypes (not part of the ABI).
#pragma once
#include <cstdint>
#include <vector>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "../../include/omok_b200.h"
#include "omk_device.cuh"

namespace omk {

constexpr int kMaxBatchPerTree = 64;  // per-tree requests per round (evaluate_batch_size)
constexpr int kNetTensors = 31;

enum ApplyMode { kApplySearch = 0, kApplyNewGame = 1, kApplyEnsure = 2 };

struct NetWeights {
    float *t[kNetTensors] = {};  // device copies in checkpoint order
    float *heads_w = nullptr;    // [512][128]: cols 0..80 policy, col 81 value, rest 0
    float *heads_b = nullptr;    // [128]
    // fp16-split tensor-core path (fc_f16.cu, tower_f16.cu): weights scaled by a power of two, then split hi/lo
    __half *fc0_wt_h16 = nullptr, *fc0_wt_l16 = nullptr;  // [512][10368] K-major
    __half *fc1_wt_h16 = nullptr, *fc1_wt_l16 = nullptr;  // [512][512]
    __half *heads_wt_h16 = nullptr, *heads_wt_l16 = nullptr;  // [128][512]: rows 0..80 policy, 81 value, rest 0
    float *fc_inv_scale = nullptr;     // [3] 2^-s of fc0, fc1, heads
    uint32_t *fc_absmax = nullptr;     // [3] max |w| bits
    uint8_t *tower16_wimg = nullptr;   // 3 x 36 KB pre-swizzled B-operand images
    float *tower16_pimg = nullptr;     // fp32 stem / bias / depthwise parameters + inverse scales
    uint32_t *tower16_absmax = nullptr;  // [9]
    bool loaded = false;
};

struct Workspace {  // evaluator request/response buffers [max_rows]; activation buffers [act_rows], allocated on first use
    int max_rows = 0;
    int act_rows = 0;
    bool act_fp32 = false;        // the fp32 buffers of the CUDA-core A/B kernels exist (act0, act1)
    NNIn *nn_in = nullptr;        // [max_rows]
    uint32_t *req_tree = nullptr; // [max_rows]
    uint32_t *req_node = nullptr; // [max_rows]
    float *P = nullptr;           // [max_rows][96]
    float *V = nullptr;           // [max_rows]
    __half *act0_h16 = nullptr, *act0_l16 = nullptr;  // [act_rows][10368] fp16 hi/lo split of the tower output == fc0's A operand
    __half *act1_h16 = nullptr, *act1_l16 = nullptr;  // [act_rows][512] fp16 hi/lo split of fc0's output == fc1's A operand
    __half *act2_h16 = nullptr, *act2_l16 = nullptr;  // [act_rows][512] fp16 hi/lo split of fc1's output == the heads' A operand
    float *act2 = nullptr;        // [act_rows][512] fc1 output (fp32: CUDA-core heads, debugging)
    float *logits = nullptr;      // [act_rows][128]
    float *act0 = nullptr;        // [act_rows][10368] fp32 tower output (CUDA-core A/B kernels only)
    float *act1 = nullptr;        // [act_rows][512]   fp32 fc0 output   (CUDA-core A/B kernels only)
    uint32_t *n_req = nullptr;    // device counter
    uint32_t *slot_base = nullptr, *slot_count = nullptr;  // [capacity_trees]
    int32_t *ids = nullptr;       // [capacity_trees] device copy of the call's id list
    int32_t *actions = nullptr;   // [capacity_trees]
    uint8_t *modes = nullptr;     // [capacity_trees]
    float *temps = nullptr;       // [capacity_trees]
    int8_t *status = nullptr;     // [capacity_trees]
    float *policy_out = nullptr;  // [capacity_trees][81]
    uint32_t *streams = nullptr;  // [capacity_trees]
};

// Replay memory on the device (replay_kernels.cu; DESIGN.md 2).  Row a (absolute: rows added since the last reset) lives
// at a % cap; logical row i (0 = oldest) is absolute row added - len + i.
struct ReplayRing {
    uint8_t *boards = nullptr;  // [cap][81]
    uint8_t *turns = nullptr;   // [cap]
    float *pi = nullptr;        // [cap][81]
    float *z = nullptr;         // [cap]
    long long cap = 0;
};
struct ReplayCounters {  // device; advanced by the per-ply commit
    long long added, len, episodes;
    uint32_t done, pad;  // arrival counter of the commit's blocks (re-armed)
};
struct Replay {
    ReplayRing ring;
    ReplayCounters *counters = nullptr;
    long long added = 0, len = 0, episodes = 0;  // host copy of *counters, refreshed by omk_selfplay_run
    // staging of the driver's unfinished games: [games][81 plies][81] boards and policies, [games] ply counts
    int stage_games = 0;  // 0: the driver does not feed the replay
    uint8_t *stage_boards = nullptr;
    float *stage_pi = nullptr;
    int32_t *stage_len = nullptr;
    cudaStream_t stream = nullptr;      // the per-ply commits
    cudaEvent_t ev_commit = nullptr;    // the last commit enqueued
};

}  // namespace omk

struct omk_prof_span {
    cudaEvent_t a, b;
    int kind;
};

struct omk_ctx {
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
    struct Scratch { void *p = nullptr; size_t cap = 0; } scratch[3];
    std::vector<uint8_t> id_seen;   // host scratch of stage_ids: duplicate detection over an id list
    int id_base = 0;                // first tree id of the lane in use when the id list is the identity

    omk::EnvRec *envs = nullptr;
    omk::TreeHdr *tree_hdrs = nullptr;
    uint8_t *tree_nodes = nullptr;   // [cap_trees][cap_nodes][kNodeBytes]
    uint16_t *remap = nullptr;       // [cap_trees][cap_nodes] compaction scratch
    uint32_t *dev_error = nullptr;   // sticky device error word
    unsigned long long *dev_sims = nullptr;  // simulations counter

    omk::NetWeights net;
    omk::Workspace ws;
    int virtual_loss = 0;           // opt-in, non-reference search mode (omk_search_set_virtual_loss); refused with the parity evaluator
    int fc0_balance = 0;            // fc0 tail balancing of the CTA-pair kernel (fc_f16.cu FcBal): 0 off (default), 1 on
    int fc0_chunk = 9;              // k-blocks of fc0 accumulated in tensor memory per drain: 9 (default) or 3 (finer, more accurate; fc_f16.cu)
    int fc0_mode = 1;               // fc0 + fc1: 1 = tcgen05 3xFP16 k_fc16 (the product path), 0 = fp32 CUDA-core k_gemm (A/B check only)
    void *fc16_state = nullptr;     // tensor maps of the fp16-split path (fc_f16.cu)
    int tower16_pairs = 0;          // resident CTA pairs of k_tower16 (0 = not queried yet)
    void *tower16_params_host = nullptr;  // host copy of the tower's fp32 parameter image (kernel argument of k_tower16)
    void *train_state = nullptr;    // trainer step workspace, Adadelta slots, optional NCCL communicator (train_kernels.cu)
    int train_n = 0;                // positions of the minibatch currently on the device (omk_train_backward)
    bool net_pack_dirty = false;    // omk_train_apply changed the fp32 weights: the tensor-core operand images (and a running self-play
                                    // driver's cached root prior) are rebuilt before the next network evaluation (ensure_packed in omk_api.cu)
    int tower_mode = 1;             // tower: 1 = tcgen05 3xFP16 k_tower16 (the product path), 0 = fp32 CUDA-core k_tower (A/B check only)

    // self-play driver state
    omk_selfplay_config sp_cfg{};
    bool sp_active = false;
    int32_t *sp_ply = nullptr;        // [n_games] device ply counters
    void *sp_buf = nullptr;           // per-game scratch (ids, actions, modes, status, cached root policy)
    // Transition ring of the self-play driver (BASELINE config 4: positions streamed to the host replay buffer): kSpRing
    // ply slots on the device, mirrored in pinned host memory; a ply's slice leaves on `sp_copy_stream` while the next
    // plies search.  Allocated by omk_selfplay_begin for sp_cfg.n_games.
    static constexpr int kSpRing = 4;
    uint8_t *sp_ring_dev = nullptr, *sp_ring_host = nullptr;  // kSpRing x [boards n*81 | policy n*81 f32 | actions n i32 | status n]
    size_t sp_ring_slot_bytes = 0;
    cudaStream_t sp_copy_stream = nullptr;
    cudaEvent_t sp_ev_rec[kSpRing][2] = {}, sp_ev_copy[kSpRing] = {};
    omk::Replay rp;                   // device replay memory (omk_replay_reset); fed by the driver when it exists at omk_selfplay_begin
    // pinned host staging
    void *pinned = nullptr;
    size_t pinned_bytes = 0;
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
void fc16_free(omk_ctx *c);
// tensor maps (CUtensorMap) of k_tower16's TMA write-out over the current workspace's act0_h16 / act0_l16
bool fc16_tower_store_maps(omk_ctx *c, const void **map_hi, const void **map_lo);
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
void train_free(omk_ctx *c);
const char *train_comm_unique_id(omk_ctx *c, uint8_t *out128);
const char *train_comm_init(omk_ctx *c, const uint8_t *id128, int nranks, int rank);
const char *train_comm_destroy(omk_ctx *c);

// tower_f16.cu
bool tower16_prepare_weights(omk_ctx *c);
bool launch_tower_f16(omk_ctx *c, const float *images_dev, int rows_bound);
void tower16_read_timing(long long *out64);

}  // namespace omk
