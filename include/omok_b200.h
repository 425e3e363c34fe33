/*
 * omok_b200.h -- C ABI of libomok_b200.so: the B200-native (sm_100a) self-play hot
 * path of AcrylicShrimp/omok-ai.  This header is the drop-in boundary: the entry
 * points are what Rust shim crates named `environment`, `mcts` and `alpha-zero`
 * would bind with `extern "C"` to keep the reference's public API for its
 * trainer (src/trainer.rs), arena (benchmark/) and GUI (gui/).  INTEGRATION.md
 * shows those bindings.  Citations are relative to the reference repository.
 *
 * Conventions
 *   - every call returns an int32 status: OMK_OK (0) or a negative OMK_ERR_*;
 *     omk_last_error() returns a thread-local message for the last failure.
 *   - plain pointers and sizes only; output buffers are caller-owned HOST memory
 *     unless the name ends in `_device`.
 *   - one context = one CUDA device = one host thread at a time (many contexts OK).
 *   - there is NO CPU fallback: without a CUDA device omk_ctx_create fails.
 *   - ids are slots in the context's pools: env ids in [0, capacity_envs),
 *     tree ids in [0, capacity_trees).  `ids == NULL` means 0..n-1.  The ids of one
 *     call must be unique (OMK_ERR_INVALID otherwise): every listed slot gets its own
 *     lane / warp, two of them on one record would race.
 *
 * Encodings (match the reference's enum declaration order)
 *   cell  : 0 Empty, 1 Black, 2 White          environment/src/lib.rs:4-9
 *   turn  : 0 Black, 1 White                   environment/src/lib.rs:21-25
 *   status: 0 InProgress, 1 Draw, 2 BlackWin, 3 WhiteWin (lib.rs:45-51);
 *           OMK_NONE (-1) is Rust's Option::None.
 */
#ifndef OMOK_B200_H
#define OMOK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define OMK_API __attribute__((visibility("default")))
#else
#define OMK_API
#endif

#define OMK_CELLS 81
#define OMK_NONE (-1)

enum {
    OMK_OK = 0,
    OMK_ERR_INVALID = -1,   /* bad argument */
    OMK_ERR_CUDA = -2,      /* CUDA runtime failure (message has the detail) */
    OMK_ERR_CAPACITY = -3,  /* a tree ran out of node slots; raise capacity_nodes */
    OMK_ERR_STATE = -4,     /* call order (e.g. search before net weights are loaded) */
    OMK_ERR_NUMERIC = -5,   /* the network produced a non-finite output (an activation beyond the fp16 range of the
                               tensor-core operand split, or non-finite weights): results of this call are invalid */
};

/* evaluator driving the search (SURVEY.md 8b/8c) */
enum {
    OMK_EVAL_NET = 0,  /* the policy/value network (alpha-zero/src/network.rs) */
    OMK_EVAL_HASH = 1, /* exact integer hash-net: bit-identical on host and device (parity/tree-only benches) */
};

/* action sampling, alpha-zero/src/agent.rs:236-241 */
enum { OMK_SAMPLE_BEST = 0, OMK_SAMPLE_BOLTZMANN = 1 };
/* EnvTurnMode, alpha-zero/src/encoder.rs:4-8 */
enum { OMK_TURN_MODE_PLAYER = 0, OMK_TURN_MODE_OPPONENT = 1 };

typedef struct omk_ctx omk_ctx;

OMK_API const char *omk_last_error(void);
OMK_API int32_t omk_version(void);

/* ---------------------------------------------------------------- context */
/* capacity_nodes: node slots per tree (<= 65535).  seed keys the specified
 * counter-based random stream that replaces the reference's thread_rng().
 * A failed create releases everything it allocated and leaves *out NULL.      */
OMK_API int32_t omk_ctx_create(int32_t device, int32_t capacity_envs, int32_t capacity_trees, int32_t capacity_nodes,
                       uint64_t seed, omk_ctx **out);
OMK_API int32_t omk_ctx_destroy(omk_ctx *ctx);
OMK_API int32_t omk_ctx_synchronize(omk_ctx *ctx);
/* the CUDA stream every kernel of this context is launched on (cudaStream_t) */
OMK_API void *omk_ctx_stream(omk_ctx *ctx);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
OMK_API int64_t omk_ctx_launch_count(omk_ctx *ctx);
/* bytes the API layer has copied host->device / device->host for this context since creation (every entry point's
 * argument and result copies, and the self-play driver's transition stream; bench.py's e2e byte counts) */
OMK_API int32_t omk_ctx_transfer_bytes(omk_ctx *ctx, int64_t *out_h2d, int64_t *out_d2h);

/* ---------------------------------------------------------------- network
 * Replaces AgentModel::{evaluate_p, evaluate_pv} (alpha-zero/src/agent_model.rs:105-134)
 * and Network::new's graph (alpha-zero/src/network.rs:51-262).                  */
#define OMK_NET_TENSORS 31
/* 31 fp32 tensors in the reference's variable / checkpoint order (network.rs:78-241):
 * conv_w[1,1,3,128] conv_b[128] {w0[1,1,128,32] b0[32] dw[3,3,32,1] pw[1,1,32,32]
 * b1[32] w2[1,1,32,128] b2[128]}x3 fc0_w[10368,512] fc0_b fc1_w[512,512] fc1_b
 * v_w[512,1] v_b[1] p_w[512,81] p_b[81]; lens = element counts (validated).     */
OMK_API int32_t omk_net_load_params(omk_ctx *ctx, const float *const *tensors, const int64_t *lens);
OMK_API int32_t omk_net_get_params(omk_ctx *ctx, float *const *tensors, const int64_t *lens);
/* random init by the reference's recipe w = N(0,1)*c (network-utils/src/lib.rs:86-92) */
OMK_API int32_t omk_net_init_random(omk_ctx *ctx, uint64_t seed);
/* evaluate_pv on n positions given as boards[n*81] cells + turns[n]; mode = EnvTurnMode.
 * out_p[n*81], out_v[n] (out_v may be NULL == evaluate_p).                      */
OMK_API int32_t omk_net_eval(omk_ctx *ctx, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                     float *out_p, float *out_v);
/* evaluate_pv on the reference's input tensor: images[n*243] f32 read as [n,9,9,3]
 * (alpha-zero/src/encoder.rs:10-46; any float values, not only {0,1}).          */
OMK_API int32_t omk_net_eval_images(omk_ctx *ctx, const float *images, int32_t n, float *out_p, float *out_v);

/* ---------------------------------------------------------------- trainer step
 * Replaces AgentModel::train (alpha-zero/src/agent_model.rs:136-168) and the training half of AgentModel::new's graph
 * (:26-103; network.rs:249-253): loss = mean((z - v)^2) + mean(softmax_cross_entropy_with_logits(logits, pi)),
 * tensorflow AdadeltaOptimizer with learning rate 0.01 (:24), rho 0.95, epsilon 1e-8 (the crate's defaults; the two
 * accumulators live in the context; the reference never saves them, omk_train_get_optimizer reads them out), one
 * minimize step, then a SECOND forward that reports the losses.  images[n*243] = encode_nn_input's tensor,
 * pi[n*81] = encode_nn_targets' policy target, z[n] = its value target (alpha-zero/src/encoder.rs:10-68); out_losses[3] = {p_loss, v_loss, loss} after the update.
 * The updated weights serve every later evaluation (omk_net_eval, the searches, the self-play driver and its cached
 * root prior): the tensor-core operand images are rebuilt by the first entry point that evaluates the network after
 * the step, not by each of an iteration's 600 steps.  fp32 CUDA kernels; correctness path, not the self-play hot path. */
OMK_API int32_t omk_train_step(omk_ctx *ctx, const float *images, const float *pi, const float *z, int32_t n, float *out_losses);
/* The same step in two halves, for callers that average the gradient themselves (data parallelism, BASELINE config 5):
 * omk_train_backward leaves the gradient of the local minibatch's mean loss in one flat DEVICE buffer (*out_count =
 * 5 643 250 floats, the 31 tensors in checkpoint order) and returns with the stream idle; omk_train_apply runs the
 * all-reduce of an attached communicator (below), Adadelta and the reporting forward.                                 */
OMK_API int32_t omk_train_backward(omk_ctx *ctx, const float *images, const float *pi, const float *z, int32_t n,
                           void **out_grads_device, int64_t *out_count);
OMK_API int32_t omk_train_apply(omk_ctx *ctx, float *out_losses);
/* host copy of the last gradient, per tensor in checkpoint order (tests); zero the Adadelta accumulators */
OMK_API int32_t omk_train_get_grads(omk_ctx *ctx, float *const *tensors, const int64_t *lens);
OMK_API int32_t omk_train_reset_optimizer(omk_ctx *ctx);
/* The Adadelta accumulators, per tensor in checkpoint order (lens as omk_net_get_params).  A context that has not
 * stepped reports zeros, which is the state its first step starts from.  With omk_net_get_params and the replay rows they
 * are what a run has to save to resume exactly (DESIGN.md 2).                                                          */
OMK_API int32_t omk_train_get_optimizer(omk_ctx *ctx, float *const *accum, float *const *accum_update, const int64_t *lens);
/* Replace them (allocating the optimizer state if it does not exist yet); the next step reads them.  Every entry must be
 * finite and >= 0 (OMK_ERR_INVALID otherwise, and nothing changes).                                                    */
OMK_API int32_t omk_train_set_optimizer(omk_ctx *ctx, const float *const *accum, const float *const *accum_update,
                                        const int64_t *lens);
/* Optional NCCL communicator for the gradient all-reduce (one rank per context / GPU; NVLink 5 / NVSwitch on a B200
 * box).  libnccl.so.2 is loaded with dlopen on first use (env OMK_NCCL_LIB overrides the name): rank 0 calls
 * omk_train_comm_unique_id and distributes the 128 bytes, every rank calls omk_train_comm_init; from then on
 * omk_train_apply / omk_train_step sum the gradients (and the reported losses) over the ranks and divide by nranks.   */
OMK_API int32_t omk_train_comm_unique_id(omk_ctx *ctx, uint8_t *out_id);
OMK_API int32_t omk_train_comm_init(omk_ctx *ctx, const uint8_t *id, int32_t nranks, int32_t rank);
OMK_API int32_t omk_train_comm_destroy(omk_ctx *ctx);

/* ---------------------------------------------------------------- diagnostics (tests / A-B runs)
 * Kernel choice for fc0 + fc1 + heads, and for the tower: 1 = the tcgen05 kernels (3-pass fp16 hi/lo split; the product
 * path and the default), 0 = the fp32 CUDA-core kernels kept in the library as an A/B check of each layer (env
 * OMK_FC0=simt / OMK_TOWER=simt at context creation).  omk_debug_get_buffer copies an intermediate activation buffer to
 * the host: 8 = tower output, 9 = fc0 output and 10 = fc1 output of the tensor-core path (hi + lo), 0 = tower output,
 * 1 = fc0 output, 2 = fc1 output, 3 = head logits of the CUDA-core path.                                                                           */
OMK_API int32_t omk_debug_set_fc0_mode(omk_ctx *ctx, int32_t mode);
OMK_API int32_t omk_debug_set_tower_mode(omk_ctx *ctx, int32_t mode);
/* k-blocks (of 64) fc0 accumulates in tensor memory between two drains into fp32 registers: 9 (default) or 3 -- the
 * tensor-core accumulator truncates, so the shorter chunk is more accurate (max relative prior error 2.1e-4 -> 1.6e-4 on
 * 20 000 positions) at +0.8 % fc0 time on large batches and slower small batches (env OMK_FC0_CHUNK=3).               */
OMK_API int32_t omk_debug_set_fc0_chunk(omk_ctx *ctx, int32_t k_blocks);
/* fc0 tail balancing (fc_f16.cu FcBal), 0 = off (default) / 1 = on (env OMK_FC0_BALANCE=1 sets the default): the CTA-pair
 * fc0 shares the K range of its last, partial wave of tiles with the otherwise idle CTA pairs; bit-identical rows either
 * way (tested).  Measured on B200 (profiles/r02_fc0_tail_balancing.md): it pays only for pools of ~256 games on one lane;
 * with two search lanes the "idle" pairs are where the other lane's kernels run, and the step gets slower. */
OMK_API int32_t omk_debug_set_fc0_balance(omk_ctx *ctx, int32_t on);
/* clock64 phase timestamps of one iteration inside k_tower16 (64 values; tests/tools/check_f16.py) */
OMK_API int32_t omk_debug_tower_timing(omk_ctx *ctx, int64_t *out64);
OMK_API int32_t omk_debug_get_buffer(omk_ctx *ctx, int32_t which, float *out, int64_t count);
/* Searches over at least `min_trees` trees run as two lanes (two streams, halves of the trees; per-tree results are
 * unaffected).  0 disables the second lane, e.g. to time kernels without cross-stream queueing (env OMK_LANE_MIN_TREES;
 * default 768).                                                                                                     */
OMK_API int32_t omk_debug_set_lane_min_trees(omk_ctx *ctx, int32_t min_trees);

/* ---------------------------------------------------------------- environment
 * Replaces environment::Environment (environment/src/lib.rs:62-193), batched.   */
OMK_API int32_t omk_env_reset(omk_ctx *ctx, const int32_t *ids, int32_t n);                      /* Environment::new  :73 */
/* place_stone (:104-166) on n envs.  out_status[n]: OMK_NONE if the cell was occupied
 * (no mutation), else the GameStatus.  out_legal[n*3]: 81-bit mask of empty cells
 * after the move (bit i of word i/32), may be NULL.                             */
OMK_API int32_t omk_env_step(omk_ctx *ctx, const int32_t *ids, const uint8_t *actions, int32_t n, int8_t *out_status,
                     uint32_t *out_legal);
/* same, on envs 0..n-1, with DEVICE pointers and no host synchronisation */
OMK_API int32_t omk_env_step_device(omk_ctx *ctx, const uint8_t *actions_device, int32_t n, int8_t *out_status_device,
                            uint32_t *out_legal_device);
/* public fields: board[n*81], turn[n], legal_move_count[n] (any may be NULL) */
OMK_API int32_t omk_env_get(omk_ctx *ctx, const int32_t *ids, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                    uint16_t *out_legal_counts);
OMK_API int32_t omk_env_set(omk_ctx *ctx, const int32_t *ids, int32_t n, const uint8_t *boards, const uint8_t *turns);
/* encode_nn_input (alpha-zero/src/encoder.rs:10-46): out[n*243] memory image */
OMK_API int32_t omk_env_encode(omk_ctx *ctx, const int32_t *ids, int32_t n, int32_t mode, float *out);
/* BASELINE config 2: envs 0..n-1 reset, then `plies` uniformly random legal moves each
 * (specified stream: stream = env id, one bounded draw per ply), auto-reset after a
 * terminal status.  Traces (HOST, may be NULL): actions[plies*n], status[plies*n].
 * One persistent launch; boards stay in registers between plies.                */
OMK_API int32_t omk_env_random_playout(omk_ctx *ctx, int32_t n, int32_t plies, uint8_t *out_actions, int8_t *out_status);

/* ---------------------------------------------------------------- tree pool
 * Replaces alpha_zero::Agent (agent.rs:10-232), ParallelMCTSExecutor::execute
 * (parallel_mcts_executor.rs:26-270), MCTSExecutor::run (mcts_executor.rs:29-255,
 * serialised) and, underneath, mcts::{MCTS, Node} (mcts/src/lib.rs, node.rs).   */
/* Agent::new for n trees; streams[n] = random-stream id per tree (NULL: stream = id) */
OMK_API int32_t omk_pool_new_games(omk_ctx *ctx, const int32_t *ids, int32_t n, const uint32_t *streams, int32_t evaluator);
/* execute(count, batch_size, epsilon, alpha, agents = ids): ceil(count/batch) rounds of
 * {batch selections+expansions per tree, one NN batch over all trees, apply+backup}. */
OMK_API int32_t omk_pool_search(omk_ctx *ctx, const int32_t *ids, int32_t n, int32_t count, int32_t batch_size,
                        float epsilon, float alpha, int32_t evaluator);
/* OPT-IN, NOT the reference's search: virtual loss inside a round (north_star's "PUCT selection with virtual loss").
 * The reference reads the statistics as they are (parallel_mcts_executor.rs:80-90), so a round's `batch_size`
 * selections of a tree usually return the same leaf; with this switch on, every pending evaluation counts as one visit
 * of value -1 along its path until its network result replaces it, which spreads a round over different lines.  Visit
 * counts then differ from the reference's by design: default OFF (env OMK_SEARCH_VIRTUAL_LOSS=1 turns it on at context
 * creation), and searches with the parity evaluator (OMK_EVAL_HASH) are refused while it is on.                       */
OMK_API int32_t omk_search_set_virtual_loss(omk_ctx *ctx, int32_t enabled);
/* Agent::sample_action: modes[n] (OMK_SAMPLE_*), temperatures[n] (Boltzmann only);
 * out_actions[n] (OMK_NONE if the policy is empty), out_policy[n*81] un-heated pi.  */
OMK_API int32_t omk_pool_sample(omk_ctx *ctx, const int32_t *ids, int32_t n, const uint8_t *modes,
                        const float *temperatures, int32_t *out_actions, float *out_policy);
/* Agent::compute_policy: out_policy[n*81], out_valid[n] (0 == None) */
OMK_API int32_t omk_pool_policy(omk_ctx *ctx, const int32_t *ids, int32_t n, float *out_policy, uint8_t *out_valid);
/* Agent::ensure_action_exists (one evaluate_p per tree, Opponent encoding) */
OMK_API int32_t omk_pool_ensure_action(omk_ctx *ctx, const int32_t *ids, const int32_t *actions, int32_t n,
                               int32_t evaluator);
/* Agent::play_action + MCTS::transition; out_status[n] may be OMK_NONE */
OMK_API int32_t omk_pool_play(omk_ctx *ctx, const int32_t *ids, const int32_t *actions, int32_t n, int8_t *out_status);
/* Agent.env of one tree */
OMK_API int32_t omk_pool_get_env(omk_ctx *ctx, int32_t id, uint8_t *out_board, uint8_t *out_turn,
                         uint16_t *out_legal_count);
/* Agent.env of n trees in one call (the root node's environment): out_boards[n*81], out_turns[n],
 * out_legal_counts[n], out_status[n] = the root's GameStatus (any may be NULL).  One launch, one synchronisation. */
OMK_API int32_t omk_pool_get_envs(omk_ctx *ctx, const int32_t *ids, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                          uint16_t *out_legal_counts, int8_t *out_status);
/* root node: n, w, p, status, policy[81] (any may be NULL) */
OMK_API int32_t omk_pool_root_stats(omk_ctx *ctx, int32_t id, uint64_t *out_n, float *out_w, float *out_p,
                            int32_t *out_status, float *out_policy);
/* root children in creation order: actions/n/w/p[81], *out_len = count */
OMK_API int32_t omk_pool_root_children(omk_ctx *ctx, int32_t id, int32_t *out_actions, uint64_t *out_n, float *out_w,
                               float *out_p, int32_t *out_len);
/* live node count and random-stream position of one tree */
OMK_API int32_t omk_pool_tree_info(omk_ctx *ctx, int32_t id, int32_t *out_nodes, uint32_t *out_rng_counter);

/* ---------------------------------------------------------------- self-play driver
 * The trainer's self-play loop (src/trainer.rs:86-204) restated as a device-resident
 * driver: n_games games, two trees per game (black agent = tree 2g, white = 2g+1),
 * per ply: search the mover's trees, sample (Boltzmann(temperature) while the game's
 * ply < temperature_threshold, then Best), play, ensure_action_exists + play on the
 * opponent trees, auto-restart finished games.  Transitions (board 81 B, pi 81 f32,
 * mover-view z placeholder, game id, ply) stream to a pinned host ring.          */
/* kernel families for profiling spans */
enum {
    OMK_K_TOWER = 0,      /* k_tower16: stem + 3 bottleneck blocks (tcgen05 kind::f16, 3-pass fp16 hi/lo split) */
    OMK_K_FC0 = 1,        /* k_fc16<10368>: fc0 10368 -> 512, CTA pairs / split-K + k_fc0_reduce (67 % of the network's flops) */
    OMK_K_FC1 = 2,        /* k_fc16<512>: fc1 512 -> 512 */
    OMK_K_HEADS = 3,      /* k_fc16<512, HEADS>: policy + value heads with tanh / softmax in the epilogue */
    OMK_K_HASH = 4,       /* k_eval_hash */
    OMK_K_SELECT = 5,     /* k_select_expand (+ request counter reset) */
    OMK_K_APPLY = 6,      /* k_apply */
    OMK_K_MOVE = 7,       /* per-ply kernels: noise, sample, record, play, ensure, restart */
    OMK_K_COUNT = 8
};

typedef struct {
    int32_t n_games;
    int32_t count;       /* evaluate_count       (src/config.rs:91) */
    int32_t batch_size;  /* evaluate_batch_size  (src/config.rs:92) */
    float epsilon;       /* :93 */
    float alpha;         /* :94 */
    float temperature;   /* :95 */
    int32_t temperature_threshold; /* :96 */
    int32_t evaluator;
} omk_selfplay_config;

typedef struct {
    int64_t simulations;    /* selection-loop iterations executed */
    int64_t positions;      /* plies played (transitions produced) */
    int64_t nn_evals;       /* positions sent through the evaluator */
    int64_t games_finished;
    int64_t h2d_bytes, d2h_bytes;
    float gpu_ms;           /* CUDA-event time of the whole call on the context stream */
    /* per-kernel-family CUDA-event time and launch count inside the call, indexed by OMK_K_*;
     * filled according to the `profile` level (0: none, 1: tower + fc0 only, 2: every family) */
    float kind_ms[OMK_K_COUNT];
    int64_t kind_launches[OMK_K_COUNT];
} omk_selfplay_stats;

OMK_API int32_t omk_selfplay_begin(omk_ctx *ctx, const omk_selfplay_config *cfg);
/* plays `plies` plies on every game; transitions stream through a pinned ring to out_* (HOST, each may
 * be NULL) in (ply, game) order: boards[plies*n*81], policy[plies*n*81], status[plies*n] */
OMK_API int32_t omk_selfplay_run(omk_ctx *ctx, int32_t plies, int32_t profile, uint8_t *out_boards, float *out_policy,
                         int8_t *out_status, int32_t *out_actions, omk_selfplay_stats *stats);
/* The model slot (0 .. 15, see omk_model_load_params; default 0, the network) whose weights the self-play driver evaluates
 * with: omk_selfplay_begin's root evaluation of all 2n trees, the search rounds of both lanes, the ensure_action_exists
 * evaluation of the other colour's trees and the cached empty-board prior that restarted games install.  A context setting
 * like omk_search_set_virtual_loss: it survives omk_selfplay_begin, and it may change while a driver is active, taking
 * effect at the driver's next evaluation.  A driver on slot s with weights W produces exactly the transitions, replay
 * rows, statistics and random streams of a driver on slot 0 with weights W.
 * The cached restart prior follows slot s only: it is re-evaluated when slot s changes (omk_model_load_params,
 * omk_model_from_net, omk_opponent_load_params / omk_opponent_from_net for s = 1; omk_net_load_params, omk_net_init_random
 * and the re-pack after training for s = 0) and, inside this call, when it switches an active driver to another slot (if
 * that evaluation fails, the call returns its error and the driver stays on its old slot).  A
 * change to any other slot -- training the network while s != 0 included -- leaves the driver's games untouched; with
 * s != 0 omk_selfplay_run does not re-pack a trained network, whatever evaluates slot 0 next does.
 * OMK_ERR_INVALID: slot outside 0 .. 15.  OMK_ERR_STATE: an active driver with OMK_EVAL_NET and an unloaded slot (nothing
 * changes).  omk_selfplay_begin and omk_selfplay_run refuse an unloaded selected slot with OMK_ERR_STATE (e.g. after a
 * load that failed halfway); OMK_EVAL_HASH never reads the slot.                                                         */
OMK_API int32_t omk_selfplay_set_model(omk_ctx *ctx, int32_t slot);

/* ---------------------------------------------------------------- replay memory
 * The trainer's replay memory (src/trainer.rs:27,206-352) kept on the device and fed by the self-play driver, so that
 * the training phase samples, encodes and steps without the host.  It holds the rows trainer.ReplayMemory would hold if
 * fed by split_episodes one ply at a time: episodes in (ply of the final move, game id) order; per episode the T original
 * transitions (board before the move, turn from the stone counts, visit policy, z), then the five symmetric copies of each
 * transition in the order rotate_90, rotate_180, rotate_270, flip_horizontal, flip_vertical; z = 1 (win of the last
 * mover) or 0 (draw) at the last ply, negated at each earlier one (a draw alternates +0.0 / -0.0).  Beyond the capacity
 * the oldest rows are dropped after each episode.  Rows are addressed by LOGICAL index: 0 is the oldest row.
 * Unfinished games are staged on the device across omk_selfplay_run calls; omk_selfplay_begin restarts every game and
 * drops them.  Storage: 410 bytes per row (246 MB at 600 000 rows) + 32.8 KB of staging per game.                      */
/* Empty the replay memory and (re)size it to `capacity` rows; 0 frees it and the driver stops feeding it.  The self-play
 * driver feeds a replay memory that exists at omk_selfplay_begin; creating one (capacity > 0 from 0) while a driver is
 * active is OMK_ERR_STATE.  Emptying one while a driver is active keeps the games' staged tails.                        */
OMK_API int32_t omk_replay_reset(omk_ctx *ctx, int64_t capacity);
/* rows held, rows added since the last reset (dropped ones included), episodes added since the last reset; as of the end
 * of the last omk_selfplay_run (any may be NULL) */
OMK_API int32_t omk_replay_info(omk_ctx *ctx, int64_t *out_len, int64_t *out_rows_added, int64_t *out_episodes);
/* rows[n] = logical indices (OMK_ERR_INVALID outside [0, len)); boards[n*81], turns[n], policy[n*81], z[n] (any may be NULL) */
OMK_API int32_t omk_replay_get(omk_ctx *ctx, const int64_t *rows, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                       float *out_policy, float *out_z);
/* Append n rows (in order, oldest first) at the newest end of the replay memory, e.g. rows omk_replay_get read out of an
 * earlier run.  Beyond the capacity the oldest rows are dropped, as after an episode; if n > capacity, only the call's last
 * `capacity` rows are kept.  rows_added grows by n and the episode count by `episodes` (>= 0); so after omk_replay_reset
 * and one append, rows_added counts from the restore and equals len.  Rows use omk_replay_get's layout, z stored bit for
 * bit (-0.0 stays -0.0).  Validation is all or nothing: cells in {0,1,2}, turn in {0,1}, policy and z finite; otherwise
 * OMK_ERR_INVALID and the memory is unchanged.  OMK_ERR_STATE if there is no replay memory.  Allowed while a self-play
 * driver is active: its next commits land after the appended rows.  Host-to-device copies only, no kernel.            */
OMK_API int32_t omk_replay_append(omk_ctx *ctx, const uint8_t *boards, const uint8_t *turns, const float *policy,
                                  const float *z, int32_t n, int64_t episodes);
/* `steps` gradient steps, each omk_train_step's sequence (forward, loss, backward, all-reduce of an attached communicator,
 * Adadelta, reporting forward) on a minibatch of m = min(n, len) rows drawn from the replay memory and encoded as
 * encode_nn_input(board, turn) in Player mode.  Step s draws its rows with Floyd's sample without replacement on the
 * specified random stream (mix64(seed ^ K), stream = (uint32_t)(first_step + s), counter from 0) (DESIGN.md 4).
 * out_losses[steps*3] = {p_loss, v_loss, loss} after each update; out_rows[steps*n] (may be NULL) = the logical rows
 * each step used, in draw order, -1 past m.  No minibatch crosses the host; one synchronisation for the whole call.
 * An absent or empty replay memory is OMK_ERR_STATE.                                                                     */
OMK_API int32_t omk_train_replay(omk_ctx *ctx, uint64_t seed, int64_t first_step, int32_t steps, int32_t n, float *out_losses,
                         int64_t *out_rows);
/* The trainer's loss terms of model slot `slot` (0 .. 15, 0 = the network) on replay rows, changing nothing: rows[n] logical
 * indices, or rows == NULL for the logical range [first, first + n).  Per row, from the policy logits l[81] and the value
 * logit of the tensor-core forward on encode_nn_input(board, turn) in Player mode (the evaluator's network, with the logits
 * kept instead of turned into probabilities; omk_debug_set_fc0_mode(ctx, 0) selects the CUDA-core heads GEMM):
 *   p_loss = -sum_a pi[a] * (l[a] - logsumexp(l))      (softmax_cross_entropy_with_logits over all 81 cells, as the trainer)
 *   v_loss = (z - tanh(value logit))^2
 *   top1   = 1 if the first maximum of l (ascending cell order) is the first maximum of pi, else 0
 * with the trainer's own loss kernel.  out_means points to a double[4] = {mean p_loss, mean v_loss, mean p_loss + mean v_loss,
 * mean top1} in fp64, in a specified order: the rows [1024 b, 1024 b + 1024) of the call are added in row order from 0.0, then
 * these block sums in ascending b, each sum divided by n; so the means depend on the rows only.  (It is declared void * because
 * the ABI's declarations stay within the scalar types the Rust bindings mirror, which have no double: pass a double[4], from
 * Rust a [f64; 4] as *mut c_void.)  out_row_p_loss[n], out_row_v_loss[n]
 * and out_row_top1[n] (each may be NULL) are the per-row terms.  Rows are read as of the end of the last omk_selfplay_run, as
 * omk_replay_info reports them; no tree, env slot, replay row, self-play or optimizer state is touched, so an active
 * self-play driver's next omk_selfplay_run is unchanged.  A network changed by training is re-packed first, as by every
 * evaluating call.  OMK_ERR_STATE: no or an empty replay memory, slot not loaded; OMK_ERR_INVALID: slot outside 0 .. 15, a row
 * outside [0, len), n < 1, out_means NULL; OMK_ERR_NUMERIC: a non-finite logit or loss.  The rows are evaluated in chunks of
 * 16 384; no host-to-device copy with rows == NULL; one synchronisation (after the first call's allocations). */
OMK_API int32_t omk_replay_score(omk_ctx *ctx, int32_t slot, const int64_t *rows, int64_t first, int32_t n, void *out_means,
                                 float *out_row_p_loss, float *out_row_v_loss, uint8_t *out_row_top1);

/* ---------------------------------------------------------------- evaluation against the naive player
 * The trainer's evaluation phase (src/trainer.rs:487-603) on the device.  The naive player (:506-537) takes the first
 * empty cell, ascending, where place_stone is terminal (win or draw) for the side to move or, with the turn flipped, for
 * the opponent; otherwise legal[below(legal_count)] over the ascending empty cells, drawn on the specified random stream
 * (mix64(seed ^ K_NAIVE), stream id, counter from 0) (DESIGN.md 4); a forced move draws nothing.                      */
/* the naive player's move for n positions: boards[n*81], turns[n]; streams[n] (NULL: i); out_actions[n] (OMK_NONE on a
 * full board); out_forced[n] (may be NULL): 1 if the move wins, blocks or fills the last cell, 0 if it was drawn at random */
OMK_API int32_t omk_naive_move(omk_ctx *ctx, const uint8_t *boards, const uint8_t *turns, int32_t n, uint64_t seed,
                               const uint32_t *streams, int32_t *out_actions, uint8_t *out_forced);
/* `episodes` games on the trees first_tree .. first_tree + episodes - 1 (tree stream = tree id; OMK_ERR_STATE if they
 * overlap an active self-play driver's trees 0 .. 2 * n_games - 1).  The naive player is Black and moves first; game g's
 * move at ply p (moves already played) uses stream g * 81 + p.  The model answers each move with ensure_action_exists +
 * play_action, and moves with execute(count, batch_size, epsilon, alpha) + sample_action(Best) + play_action.  One host
 * round trip per half-move (the live-game count); no host-to-device copy.  out_result[3] = {black (naive) wins, white
 * (model) wins, draws}; out_moves[episodes*81] (may be NULL) = each game's moves in playing order, -1 past its end;
 * out_status[episodes] (may be NULL) = final GameStatus; out_stats[4] (may be NULL) = {simulations, positions evaluated,
 * moves played, host synchronisations}; out_gpu_ms (may be NULL) = CUDA-event time of the call on the context stream. */
OMK_API int32_t omk_eval_naive(omk_ctx *ctx, int32_t episodes, int32_t first_tree, int32_t count, int32_t batch_size, float epsilon,
                               float alpha, int32_t evaluator, uint64_t seed, int32_t *out_result, int8_t *out_moves,
                               int8_t *out_status, int64_t *out_stats, float *out_gpu_ms);

/* ---------------------------------------------------------------- the opponent network and the arena
 * The opponent network: a second set of weights in the context (model slot 1), read by omk_opponent_eval, omk_match and
 * a self-play driver set to slot 1 (omk_selfplay_set_model).  Training, the searches and omk_net_* never read or change
 * it; loading it changes nothing they produce, nor what a driver on another slot produces.                             */
OMK_API int32_t omk_opponent_load_params(omk_ctx *ctx, const float *const *tensors, const int64_t *lens); /* as omk_net_load_params */
/* device-to-device copy of the network's current fp32 weights (e.g. before a training phase), images rebuilt from them;
 * OMK_ERR_STATE if no network is loaded */
OMK_API int32_t omk_opponent_from_net(omk_ctx *ctx);
OMK_API int32_t omk_opponent_eval(omk_ctx *ctx, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                                  float *out_p, float *out_v); /* omk_net_eval with the opponent's weights */
/* benchmark/src/main.rs:14-108 on the device: 2 * pairs games; games 0 .. pairs-1 the network opens (Black), games
 * pairs .. 2*pairs-1 the opponent opens.  Every move = execute(count, batch_size, epsilon, alpha) + sample_action(Best) +
 * play_action in the mover's tree, then ensure_action_exists + play_action in the other model's tree.
 * Trees: the network's tree of game j is first_tree + j, the opponent's is first_tree + 2*pairs + j; both have random
 * stream j % pairs (so arena.play_match on two contexts with this context's seed replays it game by game).  OMK_ERR_STATE
 * if they overlap an active self-play driver's trees 0 .. 2 * n_games - 1.
 * evaluator OMK_EVAL_NET: network vs opponent (both must be loaded); OMK_EVAL_HASH: the hash evaluator on both sides.
 * out_result[3] = {network wins, opponent wins, draws}; out_moves[2*pairs*81] (may be NULL) each game's moves, -1 past its
 * end; out_status[2*pairs] (may be NULL) final GameStatus; out_stats[4] (may be NULL) = {simulations, positions evaluated,
 * moves, host synchronisations}; out_gpu_ms (may be NULL).  One host round trip per half-move; no host-to-device copy. */
OMK_API int32_t omk_match(omk_ctx *ctx, int32_t pairs, int32_t first_tree, int32_t count, int32_t batch_size, float epsilon,
                          float alpha, int32_t evaluator, int32_t *out_result, int8_t *out_moves, int8_t *out_status,
                          int64_t *out_stats, float *out_gpu_ms);

/* ---------------------------------------------------------------- model slots and the tournament
 * A context holds 16 weight sets ("model slots").  Slot 0 is the network, slot 1 the opponent (omk_opponent_* are the calls
 * below with slot 1); slots 2 .. 15 are further weight sets, read only by omk_model_eval, omk_tournament and a self-play
 * driver set to them (omk_selfplay_set_model).  A slot's device buffers (about 45 MB) are allocated on its first load.
 * Slot 0 is OMK_ERR_INVALID in omk_model_load_params and omk_model_from_net: omk_net_load_params and the trainer own it. */
OMK_API int32_t omk_model_load_params(omk_ctx *ctx, int32_t slot, const float *const *tensors, const int64_t *lens); /* as omk_net_load_params */
/* device-to-device copy of the network's current fp32 weights (a snapshot); OMK_ERR_STATE if no network is loaded */
OMK_API int32_t omk_model_from_net(omk_ctx *ctx, int32_t slot);
/* device-to-host copy of slot `slot`'s (0 .. 15) 31 fp32 tensors in checkpoint order, lens as omk_net_load_params; slot 0 is
 * omk_net_get_params.  OMK_ERR_INVALID: slot out of range or a bad length; OMK_ERR_STATE: the slot is not loaded. */
OMK_API int32_t omk_model_get_params(omk_ctx *ctx, int32_t slot, float *const *tensors, const int64_t *lens);
OMK_API int32_t omk_model_eval(omk_ctx *ctx, int32_t slot, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                               float *out_p, float *out_v); /* omk_net_eval with slot `slot`'s weights; slot 0 == omk_net_eval */
/* A round-robin of omk_match over n_models (2 .. 16) distinct slots[]: P = n(n-1)/2 pairings (i, j), i < j, in lexicographic
 * order.  Pairing p is exactly omk_match(pairs, ...) with slots[i] as the network ("left") and slots[j] as the opponent
 * ("right"), on the trees first_tree + 4*pairs*p .. laid out as omk_match lays out its trees at that first tree; game g of
 * pairing p has random stream g % pairs.  Every game equals its game in that omk_match call.  At each half-move a model
 * searches all its pairings' movers as one group under its weights; the groups alternate over the two search lanes.
 * evaluator OMK_EVAL_NET: every listed slot must be loaded (OMK_ERR_STATE otherwise) and the network too, as in omk_match;
 * OMK_EVAL_HASH: the hash evaluator for every model (refused with virtual loss on).  OMK_ERR_STATE if the trees overlap an
 * active self-play driver's trees 0 .. 2 * n_games - 1.  A device error (out of node slots, a non-finite network output, a
 * refused move) ends the call at that half-move: OMK_ERR_CAPACITY, OMK_ERR_NUMERIC or OMK_ERR_STATE.
 * out_result[3*P]: per pairing {left wins, right wins, draws}; out_moves[P*2*pairs*81] and out_status[P*2*pairs] (may be
 * NULL): row p*2*pairs + g is pairing p's game g, as in omk_match; out_stats[4] (may be NULL) = {simulations, positions
 * evaluated, moves, host synchronisations}; out_gpu_ms (may be NULL).  One host round trip of 4*(n_models+1) bytes per
 * half-move; no host-to-device copy. */
OMK_API int32_t omk_tournament(omk_ctx *ctx, int32_t n_models, const int32_t *slots, int32_t pairs, int32_t first_tree, int32_t count,
                               int32_t batch_size, float epsilon, float alpha, int32_t evaluator, int32_t *out_result, int8_t *out_moves,
                               int8_t *out_status, int64_t *out_stats, float *out_gpu_ms);
/* omk_tournament with the naive player (omk_naive_move's rule, key mix64(seed ^ K_NAIVE)) as participant 0 and slots[k] as
 * participant k + 1, for n_models (1 .. 16) distinct slots: N = n_models + 1 participants, P = N(N-1)/2 pairings (a, b),
 * a < b, in lexicographic order over participants, so the first n_models are (naive, slots[k]), the naive player "left" and
 * opening games 0 .. pairs - 1.  Pairing p uses the trees first_tree + 4*pairs*p .. in omk_match's layout; in a naive
 * pairing the naive side's 2*pairs trees are reserved and never touched, and the model's tree of game g has random stream
 * g % pairs.  The naive player's move at half-move h of game g reads the board from the root of the model's tree of that
 * game and draws on stream g*81 + h; the model takes it at its next half-move (ensure_action_exists + play_action), unless
 * it ended the game.  So model-model pairing (i+1, j+1) equals pairing (i, j) of omk_tournament(slots, ...) game by game,
 * and games 0 .. pairs - 1 of (naive, slots[k]) equal omk_eval_naive(pairs, first_tree = 0, ..., seed) with slots[k] as the
 * network.  evaluator OMK_EVAL_NET: every listed slot must be loaded, and the network too (OMK_ERR_STATE otherwise).
 * Errors, outputs and accounting are omk_tournament's with N participants: one host round trip of 4*(N+1) bytes per
 * half-move, no host-to-device copy.  arena.ratings(out_result, N) then rates the naive player at 0 Elo. */
OMK_API int32_t omk_tournament_naive(omk_ctx *ctx, int32_t n_models, const int32_t *slots, int32_t pairs, int32_t first_tree,
                                     int32_t count, int32_t batch_size, float epsilon, float alpha, int32_t evaluator, uint64_t seed,
                                     int32_t *out_result, int8_t *out_moves, int8_t *out_status, int64_t *out_stats,
                                     float *out_gpu_ms);

#ifdef __cplusplus
}
#endif
#endif /* OMOK_B200_H */
