// omk_api.cu -- extern "C" boundary of libomok_b200.so (see include/omok_b200.h).
// Host-side orchestration only: pool allocation, argument staging, kernel sequencing.
// There is no CPU compute path: every operation is a CUDA kernel on the context's stream.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <utility>

#include "omk_internal.h"

using namespace omk;

static thread_local std::string g_err;
static int32_t fail(int32_t code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return fail(OMK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));             \
    } while (0)
#define CKV(call)                                                                                       \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess) g_err = std::string(#call) + ": " + cudaGetErrorString(e__);            \
    } while (0)

static const long long kLens[kNetTensors] = {
    384, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    4096, 32, 288, 1024, 32, 4096, 128,
    10368LL * 512, 512, 512 * 512, 512, 512, 1, 512 * 81, 81};


// every host <-> device copy of the API layer is counted in the context (omk_ctx_transfer_bytes; bench.py's e2e bytes)
static inline cudaError_t copy_h2d(omk_ctx *c, void *dst, const void *src, size_t bytes, cudaStream_t s) {
    c->h2d_bytes += (int64_t)bytes;
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
}
static inline cudaError_t copy_d2h(omk_ctx *c, void *dst, const void *src, size_t bytes, cudaStream_t s) {
    c->d2h_bytes += (int64_t)bytes;
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s);
}

extern "C" const char *omk_last_error(void) { return g_err.c_str(); }
extern "C" int32_t omk_version(void) { return 100; }

// ------------------------------------------------------------------ workspace
// grow-only device scratch slot i of the context (every call that uses it synchronises the stream before it returns)
template <typename T>
static int32_t scratch_dev(omk_ctx *c, int i, size_t count, T **out) {
    CK(c->scratch[i].grow(c->stream, count * sizeof(T), 4096));
    *out = reinterpret_cast<T *>(c->scratch[i].get());
    return OMK_OK;
}
#define SCRATCH(i, count, ptr)                          \
    do {                                                \
        int32_t rc__ = scratch_dev(c, (i), (count), &(ptr)); \
        if (rc__) return rc__;                          \
    } while (0)

static int32_t ensure_workspace(omk_ctx *c, int rows) {
    rows = (rows + 255) / 256 * 256;  // whole 256-row CTA-pair tiles
    Workspace &w = c->ws;
    if (rows <= w.max_rows) return OMK_OK;
    const size_t r = (size_t)rows;
    w.max_rows = 0;  // until every buffer below holds `rows` rows
    CK(w.nn_in.grow(c->stream, r));
    CK(w.req_tree.grow(c->stream, r));
    CK(w.req_node.grow(c->stream, r));
    CK(w.P.grow(c->stream, r * kRow));
    CK(w.V.grow(c->stream, r));
    CK(cudaMemsetAsync(w.nn_in, 0, w.nn_in.bytes(), c->stream));
    w.max_rows = rows;
    return OMK_OK;
}

namespace omk {
// Activation buffers of the network, sized on first use (the hash evaluator never needs them): fp16 hi/lo operands of the
// tensor-core path always; the fp32 buffers of the CUDA-core A/B kernels only once such a mode has been selected.
bool ensure_activations(omk_ctx *c, int rows) {
    Workspace &w = c->ws;
    rows = (rows + 255) / 256 * 256;
    const bool want_fp32 = c->tower_mode == 0 || c->fc0_mode == 0;
    if (rows <= w.act_rows && (!want_fp32 || w.act_fp32)) return true;
    if (rows < w.act_rows) rows = w.act_rows;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return false;
    static_cast<Activations &>(w) = Activations{};  // the old buffers go before the new ones are allocated
    Activations a;
    auto zeroed = [&](auto &b, size_t count) {  // padded tile rows read zeros, never NaNs
        return b.alloc(count) == cudaSuccess && cudaMemsetAsync(b, 0, b.bytes(), c->stream) == cudaSuccess;
    };
    const size_t r = (size_t)rows;
    // (act0: two rows of slack -- k_tower16 stores whole position triples, the last one may reach past `rows`)
    bool ok = zeroed(a.act0_h16, (r + 2) * 10368) && zeroed(a.act0_l16, (r + 2) * 10368) && zeroed(a.act1_h16, r * 512) &&
              zeroed(a.act1_l16, r * 512) && zeroed(a.act2_h16, r * 512) && zeroed(a.act2_l16, r * 512) && zeroed(a.act2, r * 512) &&
              zeroed(a.logits, r * 128);
    if (ok && want_fp32) ok = zeroed(a.act0, r * 10368) && zeroed(a.act1, r * 512);
    a.act_rows = rows;
    a.act_fp32 = want_fp32;
    if (!ok || !fc16_encode_act_maps(a)) return false;
    static_cast<Activations &>(w) = std::move(a);
    return true;
}
}  // namespace omk

// ------------------------------------------------------------------ search lanes
// RAII: lane 1 = swap the context's stream and evaluator workspace with the second lane's for the launches in scope.
struct LaneScope {
    omk_ctx *c;
    bool swapped;
    LaneScope(omk_ctx *ctx, int lane, int id_base) : c(ctx), swapped(lane == 1) {
        if (swapped) {
            std::swap(c->stream, c->lane1_stream);
            std::swap(c->ws, c->lane1_ws);
        }
        c->id_base = id_base;
    }
    ~LaneScope() {
        if (swapped) {
            std::swap(c->stream, c->lane1_stream);
            std::swap(c->ws, c->lane1_ws);
        }
        c->id_base = 0;
    }
};
// RAII: the evaluator launches in scope read the weights of model slot `slot` (either lane may evaluate any model)
struct ModelScope {
    omk_ctx *c;
    NetWeights *saved;
    ModelScope(omk_ctx *ctx, int slot) : c(ctx), saved(ctx->model) { c->model = &c->slot(slot); }
    ~ModelScope() { c->model = saved; }
};
// creates lane 1 on first use; false: this context has no second lane
static bool lane1_ready(omk_ctx *c) {
    if (!c->lane1_stream) {
        Workspace &w = c->lane1_ws;
        const size_t ct = (size_t)(c->cap_trees > 0 ? c->cap_trees : 1);
        if (cudaStreamCreateWithFlags(&c->lane1_stream, cudaStreamNonBlocking) != cudaSuccess) return false;
        bool ok = cudaEventCreateWithFlags(&c->lane_fork, cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&c->lane_join, cudaEventDisableTiming) == cudaSuccess &&
                  w.n_req.alloc(4) == cudaSuccess && w.slot_base.alloc(ct) == cudaSuccess && w.slot_count.alloc(ct) == cudaSuccess &&
                  cudaMemsetAsync(w.n_req, 0, w.n_req.bytes(), c->lane1_stream) == cudaSuccess;
        if (!ok) {
            cudaGetLastError();
            c->lane_min_trees = 0;  // no second lane on this context
            return false;
        }
    }
    return true;
}
// how many lanes a search over n trees uses
static int lanes_for(omk_ctx *c, int n) {
    if (c->lane_min_trees <= 0 || n < c->lane_min_trees || n < 2) return 1;
    return lane1_ready(c) ? 2 : 1;
}
static void lanes_fork(omk_ctx *c) {  // lane 1 starts after everything already queued on the main stream
    cudaEventRecord(c->lane_fork, c->stream);
    cudaStreamWaitEvent(c->lane1_stream, c->lane_fork, 0);
}
static void lanes_join(omk_ctx *c) {  // the main stream continues after lane 1 has drained
    cudaEventRecord(c->lane_join, c->lane1_stream);
    cudaStreamWaitEvent(c->stream, c->lane_join, 0);
}

static int32_t check_device_error(omk_ctx *c) {
    uint32_t e = 0;
    CK(copy_d2h(c, &e, c->dev_error, sizeof e, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    if (e) {
        uint32_t z = 0;
        copy_h2d(c, c->dev_error, &z, sizeof z, c->stream);
    }
    if (e & 1u) return fail(OMK_ERR_CAPACITY, "a tree ran out of node slots (capacity_nodes=" + std::to_string(c->cap_nodes) + ")");
    if (e & 4u)
        return fail(OMK_ERR_STATE, "the self-play driver sampled a move its tree refused (play_action returned None): the transition stream of this call is not usable");
    if (e & 8u) return fail(OMK_ERR_STATE, "the evaluation played a move its tree refused (play_action returned None): its result is not usable");
    if (e & 16u)
        return fail(OMK_ERR_STATE, "the match played a move a tree refused (play_action returned None), or a game's two trees fell out of step: "
                                   "its result is not usable");
    if (e & 2u)
        return fail(OMK_ERR_NUMERIC, "the network produced a non-finite policy or value (activation beyond the fp16 operand range "
                                     "of the tensor-core path, |x| >= 65504, or non-finite weights)");
    return OMK_OK;
}

// stage a host id list (or the identity) on the device; returns nullptr for identity
static int32_t stage_ids(omk_ctx *c, const int32_t *ids, int n, const int32_t **out, int limit) {
    *out = nullptr;
    if (n < 0 || n > limit) return fail(OMK_ERR_INVALID, "n out of range for the pool capacity");
    if (!ids) return OMK_OK;
    // ids must be unique: the kernels give every listed slot its own lane / warp, and two of them on one record would
    // race (n_nodes bump, edge statistics, the in-place compaction of k_play)
    if ((int)c->id_seen.size() < limit) c->id_seen.assign((size_t)limit, 0);
    bool bad = false, dup = false;
    int filled = 0;
    for (; filled < n && !bad && !dup; ++filled) {
        const int32_t id = ids[filled];
        if (id < 0 || id >= limit) bad = true;
        else if (c->id_seen[(size_t)id]) dup = true;
        else c->id_seen[(size_t)id] = 1;
    }
    for (int i = 0; i < filled; ++i)
        if (ids[i] >= 0 && ids[i] < limit) c->id_seen[(size_t)ids[i]] = 0;
    if (bad) return fail(OMK_ERR_INVALID, "id out of range");
    if (dup) return fail(OMK_ERR_INVALID, "duplicate id in the id list (ids must be unique within one call)");
    CK(copy_h2d(c, c->ws.ids, ids, sizeof(int32_t) * (size_t)n, c->stream));
    *out = c->ws.ids;
    return OMK_OK;
}

namespace omk {
bool prof_begin(omk_ctx *c, int kind, int min_level) {
    if (c->prof_level < min_level) return false;
    omk_prof_span s;
    s.kind = kind;
    for (cudaEvent_t *e : {&s.a, &s.b}) {
        if (c->prof_pool.empty()) {
            cudaEventCreate(e);
        } else {
            *e = c->prof_pool.back();
            c->prof_pool.pop_back();
        }
    }
    cudaEventRecord(s.a, c->stream);
    c->prof_spans.push_back(s);
    return true;
}
void prof_end(omk_ctx *c, bool opened) {
    if (opened) cudaEventRecord(c->prof_spans.back().b, c->stream);
}
}  // namespace omk

// false: the evaluator did not run to the end of its launch sequence (ws.P / ws.V are stale): the caller returns
// OMK_ERR_CUDA WITHOUT launching k_apply, which would write those rows into tree policies and back up garbage values
static bool run_evaluator(omk_ctx *c, int evaluator, int rows_bound) {
    if (evaluator == OMK_EVAL_HASH) {
        const bool sp = prof_begin(c, OMK_K_HASH, 2);
        launch_eval_hash(c, rows_bound);
        prof_end(c, sp);
        return true;
    }
    return net_forward(c, nullptr, rows_bound);
}
#define RUN_EVAL(c, evaluator, rows)                                                                                   \
    do {                                                                                                               \
        if (!run_evaluator((c), (evaluator), (rows)))                                                                  \
            return fail(OMK_ERR_CUDA, "the evaluator failed to launch (see stderr); no result was applied to the trees"); \
    } while (0)

static int32_t weights_changed(omk_ctx *c);
// The trainer's 600 updates per iteration do not evaluate the network in between (the step's own forward passes read the fp32
// weights), so omk_train_apply only marks the tensor-core operand images stale; they are rebuilt here, on the main stream and
// before any search lane forks, by every entry point that is about to evaluate the network.
static int32_t ensure_packed(omk_ctx *c) {
    if (!c->net_pack_dirty) return OMK_OK;
    const int32_t rc = weights_changed(c);
    if (rc == OMK_OK) c->net_pack_dirty = false;  // a failed rebuild is retried (and reported again) by the next evaluation
    return rc;
}

static int32_t check_evaluator(omk_ctx *c, int evaluator) {
    if (evaluator != OMK_EVAL_NET && evaluator != OMK_EVAL_HASH) return fail(OMK_ERR_INVALID, "unknown evaluator");
    if (evaluator == OMK_EVAL_HASH && c->virtual_loss)
        return fail(OMK_ERR_STATE, "virtual loss is a non-reference search mode: it is refused with the parity evaluator (OMK_EVAL_HASH)");
    if (evaluator == OMK_EVAL_NET && !c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    if (evaluator == OMK_EVAL_NET) return ensure_packed(c);
    return OMK_OK;
}

// ------------------------------------------------------------------ context
omk_ctx::~omk_ctx() {
    const cudaStream_t streams[] = {stream, lane1_stream, sp_copy_stream, rp.stream};
    for (cudaStream_t s : streams)
        if (s) cudaStreamSynchronize(s);
    for (cudaEvent_t e : prof_pool) cudaEventDestroy(e);
    for (const omk_prof_span &s : prof_spans) {
        cudaEventDestroy(s.a);
        cudaEventDestroy(s.b);
    }
    for (int i = 0; i < kSpRing; ++i)
        for (cudaEvent_t e : {sp_ev_rec[i][0], sp_ev_rec[i][1], sp_ev_copy[i]})
            if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : {ev0, ev1, lane_fork, lane_join, rp.ev_commit})
        if (e) cudaEventDestroy(e);
    for (cudaStream_t s : streams)
        if (s) cudaStreamDestroy(s);
}  // the members' destructors release the buffers

static int32_t ctx_create(int32_t device, int32_t capacity_envs, int32_t capacity_trees, int32_t capacity_nodes, uint64_t seed,
                          std::unique_ptr<omk_ctx> &ctx) {
    if (capacity_envs < 0 || capacity_trees < 0 || capacity_nodes < 2 || capacity_nodes > 65535)
        return fail(OMK_ERR_INVALID, "bad capacity (capacity_nodes must be in [2, 65535])");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(OMK_ERR_CUDA, "no CUDA device: libomok_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(OMK_ERR_INVALID, "device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(OMK_ERR_CUDA, "libomok_b200 is built for sm_100a (B200) only");

    ctx.reset(new omk_ctx());
    omk_ctx *c = ctx.get();
    c->device = device;
    c->n_sms = prop.multiProcessorCount;
    c->cap_envs = capacity_envs;
    c->cap_trees = capacity_trees;
    c->cap_nodes = capacity_nodes;
    c->seed = seed;
    auto parse_mode = [](const char *m) { return strcmp(m, "simt") == 0 ? 0 : 1; };
    if (const char *m = getenv("OMK_FC0")) c->fc0_mode = parse_mode(m);
    if (const char *m = getenv("OMK_TOWER")) c->tower_mode = parse_mode(m);
    if (const char *m = getenv("OMK_LANE_MIN_TREES")) c->lane_min_trees = atoi(m);
    if (const char *m = getenv("OMK_FC0_CHUNK")) c->fc0_chunk = atoi(m) == 3 ? 3 : 9;
    if (const char *m = getenv("OMK_FC0_BALANCE")) c->fc0_balance = atoi(m) != 0;
    if (const char *m = getenv("OMK_SEARCH_VIRTUAL_LOSS")) c->virtual_loss = atoi(m) != 0;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&c->ev0));
    CK(cudaEventCreate(&c->ev1));
    const int ce = capacity_envs > 0 ? capacity_envs : 1, ct = capacity_trees > 0 ? capacity_trees : 1;
    CK(c->envs.alloc((size_t)ce));
    CK(c->tree_hdrs.alloc((size_t)ct));
    CK(c->tree_nodes.alloc((size_t)ct * (size_t)capacity_nodes * kNodeBytes));
    CK(c->remap.alloc((size_t)ct * (size_t)capacity_nodes));
    CK(c->dev_error.alloc(1));
    CK(c->dev_sims.alloc(2));
    CK(cudaMemsetAsync(c->dev_error, 0, c->dev_error.bytes(), c->stream));
    CK(cudaMemsetAsync(c->dev_sims, 0, c->dev_sims.bytes(), c->stream));
    CK(cudaMemsetAsync(c->tree_hdrs, 0, c->tree_hdrs.bytes(), c->stream));
    CK(cudaMemsetAsync(c->envs, 0, c->envs.bytes(), c->stream));
    Workspace &w = c->ws;
    const int cm = ce > ct ? ce : ct;
    CK(w.n_req.alloc(4));
    CK(cudaMemsetAsync(w.n_req, 0, w.n_req.bytes(), c->stream));
    CK(w.slot_base.alloc((size_t)ct));
    CK(w.slot_count.alloc((size_t)ct));
    CK(w.ids.alloc((size_t)cm));
    CK(w.actions.alloc((size_t)cm));
    CK(w.modes.alloc((size_t)cm));
    CK(w.temps.alloc((size_t)cm));
    CK(w.status.alloc((size_t)cm));
    CK(w.policy_out.alloc((size_t)ct * kCells));
    CK(w.streams.alloc((size_t)ct));
    for (int i = 0; i < kNetTensors; ++i) CK(c->net.t[i].alloc((size_t)kLens[i]));
    CK(c->net.heads_w.alloc(512 * 128));
    CK(c->net.heads_b.alloc(128));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_ctx_create(int32_t device, int32_t capacity_envs, int32_t capacity_trees, int32_t capacity_nodes,
                                  uint64_t seed, omk_ctx **out) {
    if (!out) return fail(OMK_ERR_INVALID, "out is NULL");
    *out = nullptr;
    std::unique_ptr<omk_ctx> c;
    const int32_t rc = ctx_create(device, capacity_envs, capacity_trees, capacity_nodes, seed, c);
    if (rc != OMK_OK) {
        c.reset();           // releases whatever was allocated
        cudaGetLastError();  // the failed call's error must not surface in a later call
        return rc;
    }
    *out = c.release();
    return OMK_OK;
}

extern "C" int32_t omk_ctx_destroy(omk_ctx *c) {
    if (!c) return OMK_OK;
    cudaSetDevice(c->device);
    delete c;
    return OMK_OK;
}

extern "C" int32_t omk_ctx_synchronize(omk_ctx *c) {
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}
extern "C" void *omk_ctx_stream(omk_ctx *c) { return (void *)c->stream; }
extern "C" int64_t omk_ctx_launch_count(omk_ctx *c) { return c->launches; }
extern "C" int32_t omk_ctx_transfer_bytes(omk_ctx *c, int64_t *out_h2d, int64_t *out_d2h) {
    if (out_h2d) *out_h2d = c->h2d_bytes;
    if (out_d2h) *out_d2h = c->d2h_bytes;
    return OMK_OK;
}

// ------------------------------------------------------------------ network
static int32_t sp_refresh_root_policy(omk_ctx *c);  // self-play driver: re-evaluate the cached empty-board prior

extern "C" int32_t omk_net_load_params(omk_ctx *c, const float *const *tensors, const int64_t *lens) {
    CK(cudaSetDevice(c->device));
    for (int i = 0; i < kNetTensors; ++i)
        if (!tensors[i] || lens[i] != kLens[i])
            return fail(OMK_ERR_INVALID, "tensor " + std::to_string(i) + ": expected " + std::to_string(kLens[i]) + " elements");
    for (int i = 0; i < kNetTensors; ++i)
        CK(copy_h2d(c, c->net.t[i], tensors[i], sizeof(float) * (size_t)kLens[i], c->stream));
    c->net_pack_dirty = false;  // rebuilt right here
    net_pack_heads(c);
    if (!fc16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split fc weight preparation failed");
    if (!tower16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split tower weight preparation failed");
    CK(cudaStreamSynchronize(c->stream));
    c->net.loaded = true;
    return sp_refresh_root_policy(c);
}
extern "C" int32_t omk_net_get_params(omk_ctx *c, float *const *tensors, const int64_t *lens) {
    CK(cudaSetDevice(c->device));
    if (!c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    for (int i = 0; i < kNetTensors; ++i)
        if (!tensors[i] || lens[i] != kLens[i]) return fail(OMK_ERR_INVALID, "bad tensor length");
    for (int i = 0; i < kNetTensors; ++i)
        CK(copy_d2h(c, tensors[i], c->net.t[i], sizeof(float) * (size_t)kLens[i], c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}
extern "C" int32_t omk_net_init_random(omk_ctx *c, uint64_t seed) {
    CK(cudaSetDevice(c->device));
    launch_net_init_random(c, seed);
    c->net_pack_dirty = false;  // rebuilt right here
    net_pack_heads(c);
    if (!fc16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split fc weight preparation failed");
    if (!tower16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split tower weight preparation failed");
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    c->net.loaded = true;
    return sp_refresh_root_policy(c);
}

// slot: the model whose weights evaluate (omk_model_eval); only the network's (slot 0) are changed by training steps
static int32_t net_eval_common(omk_ctx *c, int n, const float *images_dev, float *out_p, float *out_v, int slot = 0) {
    if (slot == 0) {
        int32_t rc_p = ensure_packed(c);
        if (rc_p) return rc_p;
    }
    ModelScope scope(c, slot);
    if (!net_forward(c, images_dev, n)) return fail(OMK_ERR_CUDA, "the network forward failed to launch (see stderr)");
    // P rows are padded to 96 floats on the device; compact on the way out
    CK(cudaMemcpy2DAsync(out_p, sizeof(float) * kCells, c->ws.P, sizeof(float) * kRow, sizeof(float) * kCells, (size_t)n,
                         cudaMemcpyDeviceToHost, c->stream));
    c->d2h_bytes += (int64_t)sizeof(float) * kCells * n;
    if (out_v) CK(copy_d2h(c, out_v, c->ws.V, sizeof(float) * (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return check_device_error(c);  // OMK_ERR_NUMERIC when the network produced a non-finite output
}

static std::string slot_name(int slot) {
    return slot == 0 ? "network" : (slot == 1 ? "opponent" : "model slot " + std::to_string(slot));
}
static int32_t eval_boards(omk_ctx *c, int slot, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                           float *out_p, float *out_v) {
    CK(cudaSetDevice(c->device));
    if (!c->slot(slot).loaded) return fail(OMK_ERR_STATE, slot_name(slot) + " weights not loaded");
    if (n < 0 || !boards || !turns || !out_p) return fail(OMK_ERR_INVALID, "bad arguments");
    if (n == 0) return OMK_OK;
    int32_t rc = ensure_workspace(c, n);
    if (rc) return rc;
    uint8_t *d_boards = nullptr, *d_turns = nullptr;
    SCRATCH(0, (size_t)n * kCells, d_boards);
    SCRATCH(1, (size_t)n, d_turns);
    CK(copy_h2d(c, d_boards, boards, (size_t)n * kCells, c->stream));
    CK(copy_h2d(c, d_turns, turns, (size_t)n, c->stream));
    launch_pack_boards(c, d_boards, d_turns, n, mode);
    return net_eval_common(c, n, nullptr, out_p, out_v, slot);
}
extern "C" int32_t omk_net_eval(omk_ctx *c, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                                float *out_p, float *out_v) {
    return eval_boards(c, 0, boards, turns, n, mode, out_p, out_v);
}

extern "C" int32_t omk_net_eval_images(omk_ctx *c, const float *images, int32_t n, float *out_p, float *out_v) {
    CK(cudaSetDevice(c->device));
    if (!c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    if (n < 0 || !images || !out_p) return fail(OMK_ERR_INVALID, "bad arguments");
    if (n == 0) return OMK_OK;
    int32_t rc = ensure_workspace(c, n);
    if (rc) return rc;
    float *d_img = nullptr;
    SCRATCH(0, (size_t)n * 243, d_img);
    CK(copy_h2d(c, d_img, images, sizeof(float) * (size_t)n * 243, c->stream));
    const uint32_t nn = (uint32_t)n;
    CK(copy_h2d(c, c->ws.n_req, &nn, sizeof nn, c->stream));
    return net_eval_common(c, n, d_img, out_p, out_v);
}

// ------------------------------------------------------------------ trainer step (AgentModel::train)
// after the optimizer changed the fp32 tensors: re-pack the heads, re-split the tensor-core operands, refresh the
// self-play driver's cached root prior -- exactly what omk_net_load_params does after its copies
static int32_t weights_changed(omk_ctx *c) {
    net_pack_heads(c);
    if (!fc16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split fc weight preparation failed");
    if (!tower16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split tower weight preparation failed");
    CK(cudaStreamSynchronize(c->stream));
    return sp_refresh_root_policy(c);
}

static int32_t train_backward_impl(omk_ctx *c, const float *images, const float *pi, const float *z, int32_t n,
                                   void **out_grads_device, int64_t *out_count, bool sync) {
    CK(cudaSetDevice(c->device));
    if (!c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    if (n < 1 || !images || !pi || !z) return fail(OMK_ERR_INVALID, "bad arguments");
    float *g = nullptr;
    c->train_n = 0;
    if (const char *e = train_backward_step(c, images, pi, z, n, &g)) return fail(OMK_ERR_CUDA, std::string("omk_train_backward: ") + e);
    if (sync) {  // the caller may all-reduce the gradient buffer on its own stream (the fused step stays on this one)
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaGetLastError());
    }
    c->train_n = n;
    if (out_grads_device) *out_grads_device = g;
    if (out_count) *out_count = 5643250;
    return OMK_OK;
}

extern "C" int32_t omk_train_backward(omk_ctx *c, const float *images, const float *pi, const float *z, int32_t n,
                                      void **out_grads_device, int64_t *out_count) {
    return train_backward_impl(c, images, pi, z, n, out_grads_device, out_count, true);
}

extern "C" int32_t omk_train_apply(omk_ctx *c, float *out_losses) {
    CK(cudaSetDevice(c->device));
    if (c->train_n < 1) return fail(OMK_ERR_STATE, "omk_train_backward has not produced a gradient");
    if (const char *e = train_apply_step(c)) return fail(OMK_ERR_CUDA, std::string("omk_train_apply: ") + e);
    c->net_pack_dirty = true;  // the operand images of the tensor-core path follow before the next evaluation (ensure_packed)
    float l[3] = {0, 0, 0};
    if (const char *e = train_report_losses(c, c->train_n, l)) return fail(OMK_ERR_CUDA, std::string("omk_train_apply: ") + e);
    c->train_n = 0;  // one gradient, one update
    if (!(l[2] == l[2]) || l[2] > 3.0e38f) return fail(OMK_ERR_NUMERIC, "the training loss is not finite");
    if (out_losses) memcpy(out_losses, l, sizeof l);
    return OMK_OK;
}

extern "C" int32_t omk_train_step(omk_ctx *c, const float *images, const float *pi, const float *z, int32_t n, float *out_losses) {
    int32_t rc = train_backward_impl(c, images, pi, z, n, nullptr, nullptr, false);
    if (rc) return rc;
    return omk_train_apply(c, out_losses);
}

extern "C" int32_t omk_train_get_grads(omk_ctx *c, float *const *tensors, const int64_t *lens) {
    CK(cudaSetDevice(c->device));
    const float *g = train_grad_buffer(c);
    if (!g) return fail(OMK_ERR_STATE, "omk_train_backward has not run");
    long long off = 0;
    for (int i = 0; i < kNetTensors; ++i) {
        if (!tensors[i] || lens[i] != kLens[i]) return fail(OMK_ERR_INVALID, "bad tensor length");
        CK(copy_d2h(c, tensors[i], g + off, sizeof(float) * (size_t)kLens[i], c->stream));
        off += kLens[i];
    }
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_train_reset_optimizer(omk_ctx *c) {
    CK(cudaSetDevice(c->device));
    train_reset_optimizer(c);
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_train_comm_unique_id(omk_ctx *c, uint8_t *out_id) {
    if (!out_id) return fail(OMK_ERR_INVALID, "out_id is NULL");
    if (const char *e = train_comm_unique_id(c, out_id)) return fail(OMK_ERR_STATE, std::string("NCCL: ") + e);
    return OMK_OK;
}
extern "C" int32_t omk_train_comm_init(omk_ctx *c, const uint8_t *id, int32_t nranks, int32_t rank) {
    CK(cudaSetDevice(c->device));
    if (!id || nranks < 1 || rank < 0 || rank >= nranks) return fail(OMK_ERR_INVALID, "bad communicator arguments");
    if (const char *e = train_comm_init(c, id, nranks, rank)) return fail(OMK_ERR_STATE, std::string("NCCL: ") + e);
    return OMK_OK;
}
extern "C" int32_t omk_train_comm_destroy(omk_ctx *c) {
    CK(cudaSetDevice(c->device));
    train_comm_destroy(c);
    return OMK_OK;
}

// ------------------------------------------------------------------ diagnostics
extern "C" int32_t omk_debug_set_fc0_mode(omk_ctx *c, int32_t mode) {
    if (mode != 0 && mode != 1) return fail(OMK_ERR_INVALID, "fc0 mode must be 1 (tcgen05 3xFP16) or 0 (fp32 CUDA cores, A/B check)");
    c->fc0_mode = mode;
    return OMK_OK;
}
extern "C" int32_t omk_debug_set_tower_mode(omk_ctx *c, int32_t mode) {
    if (mode != 0 && mode != 1) return fail(OMK_ERR_INVALID, "tower mode must be 1 (tcgen05 3xFP16) or 0 (fp32 CUDA cores, A/B check)");
    c->tower_mode = mode;
    return OMK_OK;
}
extern "C" int32_t omk_debug_set_fc0_balance(omk_ctx *c, int32_t on) {
    if (on != 0 && on != 1) return fail(OMK_ERR_INVALID, "fc0 balance must be 0 or 1");
    c->fc0_balance = on;
    return OMK_OK;
}
extern "C" int32_t omk_debug_set_fc0_chunk(omk_ctx *c, int32_t k_blocks) {
    if (k_blocks != 3 && k_blocks != 9) return fail(OMK_ERR_INVALID, "fc0 chunk must be 9 (default) or 3 (finer accumulation)");
    CK(cudaStreamSynchronize(c->stream));
    c->fc0_chunk = k_blocks;
    return OMK_OK;
}
extern "C" int32_t omk_debug_set_lane_min_trees(omk_ctx *c, int32_t min_trees) {
    if (min_trees < 0) return fail(OMK_ERR_INVALID, "min_trees < 0");
    c->lane_min_trees = min_trees;
    return OMK_OK;
}
extern "C" int32_t omk_debug_tower_timing(omk_ctx *c, int64_t *out64) {
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    tower16_read_timing(reinterpret_cast<long long *>(out64));
    return OMK_OK;
}
extern "C" int32_t omk_debug_get_buffer(omk_ctx *c, int32_t which, float *out, int64_t count) {
    CK(cudaSetDevice(c->device));
    if (which >= 8 && which <= 10) {  // fp16-split buffers, reconstructed as hi + lo: 8 = tower, 9 = fc0, 10 = fc1 output
        if (!out || count < 0) return fail(OMK_ERR_INVALID, "bad buffer");
        const __half *hi = which == 8 ? c->ws.act0_h16 : which == 9 ? c->ws.act1_h16 : c->ws.act2_h16;
        const __half *lo = which == 8 ? c->ws.act0_l16 : which == 9 ? c->ws.act1_l16 : c->ws.act2_l16;
        if (!hi || !lo) return fail(OMK_ERR_STATE, "the tensor-core activation buffers do not exist yet (no network call so far)");
        float *tmp = nullptr;
        SCRATCH(0, (size_t)(count > 0 ? count : 1), tmp);
        launch_split16_to_f32(c, hi, lo, tmp, count);
        CK(copy_d2h(c, out, tmp, sizeof(float) * (size_t)count, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return OMK_OK;
    }
    const float *src = which == 0 ? c->ws.act0 : which == 1 ? c->ws.act1 : which == 2 ? c->ws.act2 : which == 3 ? c->ws.logits.get() : nullptr;
    if (!src || !out || count < 0) return fail(OMK_ERR_INVALID, "bad buffer id");
    CK(copy_d2h(c, out, src, sizeof(float) * (size_t)count, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

// ------------------------------------------------------------------ environment
extern "C" int32_t omk_env_reset(omk_ctx *c, const int32_t *ids, int32_t n) {
    CK(cudaSetDevice(c->device));
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_envs);
    if (rc) return rc;
    launch_env_reset(c, d_ids, n);
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_env_step(omk_ctx *c, const int32_t *ids, const uint8_t *actions, int32_t n, int8_t *out_status,
                                uint32_t *out_legal) {
    CK(cudaSetDevice(c->device));
    if (!actions) return fail(OMK_ERR_INVALID, "actions is NULL");
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_envs);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    uint8_t *d_act = nullptr;
    int8_t *d_st = nullptr;
    uint32_t *d_legal = nullptr;
    SCRATCH(0, (size_t)n, d_act);
    SCRATCH(1, (size_t)n, d_st);
    if (out_legal) SCRATCH(2, 3 * (size_t)n, d_legal);
    CK(copy_h2d(c, d_act, actions, (size_t)n, c->stream));
    launch_env_step(c, d_ids, d_act, n, d_st, d_legal);
    if (out_status) CK(copy_d2h(c, out_status, d_st, (size_t)n, c->stream));
    if (out_legal) CK(copy_d2h(c, out_legal, d_legal, sizeof(uint32_t) * 3 * (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

extern "C" int32_t omk_env_step_device(omk_ctx *c, const uint8_t *actions_device, int32_t n, int8_t *out_status_device,
                                       uint32_t *out_legal_device) {
    if (n < 0 || n > c->cap_envs) return fail(OMK_ERR_INVALID, "n exceeds capacity_envs");
    launch_env_step(c, nullptr, actions_device, n, out_status_device, out_legal_device);
    return OMK_OK;
}

extern "C" int32_t omk_env_get(omk_ctx *c, const int32_t *ids, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                               uint16_t *out_legal_counts) {
    CK(cudaSetDevice(c->device));
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_envs);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    uint8_t *d_b = nullptr, *d_t = nullptr;
    uint16_t *d_l = nullptr;
    SCRATCH(0, (size_t)n * kCells, d_b);
    SCRATCH(1, (size_t)n, d_t);
    SCRATCH(2, (size_t)n, d_l);
    launch_env_get(c, d_ids, n, d_b, d_t, d_l);
    if (out_boards) CK(copy_d2h(c, out_boards, d_b, (size_t)n * kCells, c->stream));
    if (out_turns) CK(copy_d2h(c, out_turns, d_t, (size_t)n, c->stream));
    if (out_legal_counts) CK(copy_d2h(c, out_legal_counts, d_l, sizeof(uint16_t) * (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_env_set(omk_ctx *c, const int32_t *ids, int32_t n, const uint8_t *boards, const uint8_t *turns) {
    CK(cudaSetDevice(c->device));
    if (!boards || !turns) return fail(OMK_ERR_INVALID, "NULL argument");
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_envs);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    uint8_t *d_b = nullptr, *d_t = nullptr;
    SCRATCH(0, (size_t)n * kCells, d_b);
    SCRATCH(1, (size_t)n, d_t);
    CK(copy_h2d(c, d_b, boards, (size_t)n * kCells, c->stream));
    CK(copy_h2d(c, d_t, turns, (size_t)n, c->stream));
    launch_env_set(c, d_ids, n, d_b, d_t);
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_env_encode(omk_ctx *c, const int32_t *ids, int32_t n, int32_t mode, float *out) {
    CK(cudaSetDevice(c->device));
    if (n == 0) return OMK_OK;
    if (!out) return fail(OMK_ERR_INVALID, "out is NULL");
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_envs);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    float *d_o = nullptr;
    SCRATCH(0, 243 * (size_t)n, d_o);
    launch_env_encode(c, d_ids, n, mode, d_o);
    CK(copy_d2h(c, out, d_o, sizeof(float) * 243 * (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_env_random_playout(omk_ctx *c, int32_t n, int32_t plies, uint8_t *out_actions, int8_t *out_status) {
    CK(cudaSetDevice(c->device));
    if (n < 0 || n > c->cap_envs || plies < 0) return fail(OMK_ERR_INVALID, "bad arguments");
    if (n == 0 || plies == 0) return OMK_OK;
    uint8_t *d_a = nullptr;
    int8_t *d_s = nullptr;
    const size_t tot = (size_t)n * (size_t)plies;
    if (out_actions) SCRATCH(0, tot, d_a);
    if (out_status) SCRATCH(1, tot, d_s);
    launch_env_playout(c, n, plies, d_a, d_s);
    if (out_actions) CK(copy_d2h(c, out_actions, d_a, tot, c->stream));
    if (out_status) CK(copy_d2h(c, out_status, d_s, tot, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

// ------------------------------------------------------------------ tree pool
extern "C" int32_t omk_pool_new_games(omk_ctx *c, const int32_t *ids, int32_t n, const uint32_t *streams, int32_t evaluator) {
    CK(cudaSetDevice(c->device));
    int32_t rc = check_evaluator(c, evaluator);
    if (rc) return rc;
    const int32_t *d_ids;
    rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    rc = ensure_workspace(c, n);
    if (rc) return rc;
    const uint32_t *d_streams = nullptr;
    if (streams) {
        CK(copy_h2d(c, c->ws.streams, streams, sizeof(uint32_t) * (size_t)n, c->stream));
        d_streams = c->ws.streams;
    }
    launch_reset_requests(c);
    launch_new_games(c, d_ids, n, d_streams, nullptr, nullptr);
    RUN_EVAL(c, evaluator, n);
    launch_apply(c, d_ids, n, kApplyNewGame);
    return check_device_error(c);
}

// round r of execute(count, batch_size, epsilon, alpha) on the n trees of ids (nullptr: the lane's slice), on the lane in use
static int32_t search_round(omk_ctx *c, const int32_t *ids, int n, int r, int batch_size, float epsilon, float alpha, int evaluator) {
    if (r == 0) launch_root_noise(c, ids, n, epsilon, alpha);
    launch_reset_requests(c);
    launch_select_expand(c, ids, n, batch_size);
    RUN_EVAL(c, evaluator, n * batch_size);
    launch_apply(c, ids, n, kApplySearch);
    return OMK_OK;
}

// execute(count, batch_size, epsilon, alpha) on the n >= 1 trees of d_ids (nullptr: 0..n-1), queued on the context stream;
// the caller checks the device error word
static int32_t search_rounds(omk_ctx *c, const int32_t *d_ids, int n, int count, int batch_size, float epsilon, float alpha,
                             int evaluator) {
    const int rounds = (count + batch_size - 1) / batch_size;  // parallel_mcts_executor.rs:39-42,207
    // large searches run as two lanes (halves of the id list) on two streams: per-tree results do not depend on the split
    const int lanes = lanes_for(c, n);
    const int lane_n[2] = {lanes == 2 ? (n + 1) / 2 : n, lanes == 2 ? n / 2 : 0};
    const int lane_first[2] = {0, lane_n[0]};
    for (int l = 0; l < lanes; ++l) {
        LaneScope scope(c, l, 0);
        int32_t rc = ensure_workspace(c, lane_n[l] * batch_size);
        if (rc) return rc;
    }
    if (lanes == 2) lanes_fork(c);
    for (int r = 0; r < rounds; ++r) {
        for (int l = 0; l < lanes; ++l) {
            LaneScope scope(c, l, lane_first[l]);
            const int32_t *ids_l = d_ids ? d_ids + lane_first[l] : nullptr;
            const int32_t rc = search_round(c, ids_l, lane_n[l], r, batch_size, epsilon, alpha, evaluator);
            if (rc) return rc;
        }
    }
    if (lanes == 2) lanes_join(c);
    return OMK_OK;
}

extern "C" int32_t omk_pool_search(omk_ctx *c, const int32_t *ids, int32_t n, int32_t count, int32_t batch_size, float epsilon,
                                   float alpha, int32_t evaluator) {
    CK(cudaSetDevice(c->device));
    int32_t rc = check_evaluator(c, evaluator);
    if (rc) return rc;
    if (batch_size < 1 || batch_size > kMaxBatchPerTree) return fail(OMK_ERR_INVALID, "batch_size must be in [1, 64]");
    if (count < 0) return fail(OMK_ERR_INVALID, "count < 0");
    const int32_t *d_ids;
    rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0 || count == 0) return OMK_OK;
    rc = search_rounds(c, d_ids, n, count, batch_size, epsilon, alpha, evaluator);
    if (rc) return rc;
    return check_device_error(c);
}

extern "C" int32_t omk_search_set_virtual_loss(omk_ctx *c, int32_t enabled) {
    CK(cudaStreamSynchronize(c->stream));
    c->virtual_loss = enabled != 0;
    return OMK_OK;
}

extern "C" int32_t omk_pool_sample(omk_ctx *c, const int32_t *ids, int32_t n, const uint8_t *modes, const float *temperatures,
                                   int32_t *out_actions, float *out_policy) {
    CK(cudaSetDevice(c->device));
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    const uint8_t *d_modes = nullptr;
    const float *d_temps = nullptr;
    if (modes) {
        bool any_boltz = false;
        for (int i = 0; i < n; ++i) any_boltz |= modes[i] == OMK_SAMPLE_BOLTZMANN;
        if (any_boltz && !temperatures) return fail(OMK_ERR_INVALID, "Boltzmann sampling needs temperatures");
        CK(copy_h2d(c, c->ws.modes, modes, (size_t)n, c->stream));
        d_modes = c->ws.modes;
        if (temperatures) {
            CK(copy_h2d(c, c->ws.temps, temperatures, sizeof(float) * (size_t)n, c->stream));
            d_temps = c->ws.temps;
        }
    }
    launch_sample(c, d_ids, n, d_modes, d_temps, c->ws.actions, c->ws.policy_out, nullptr);
    if (out_actions) CK(copy_d2h(c, out_actions, c->ws.actions, sizeof(int32_t) * (size_t)n, c->stream));
    if (out_policy) CK(copy_d2h(c, out_policy, c->ws.policy_out, sizeof(float) * kCells * (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

extern "C" int32_t omk_pool_policy(omk_ctx *c, const int32_t *ids, int32_t n, float *out_policy, uint8_t *out_valid) {
    CK(cudaSetDevice(c->device));
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    launch_sample(c, d_ids, n, nullptr, nullptr, nullptr, c->ws.policy_out, c->ws.modes);
    if (out_policy) CK(copy_d2h(c, out_policy, c->ws.policy_out, sizeof(float) * kCells * (size_t)n, c->stream));
    if (out_valid) CK(copy_d2h(c, out_valid, c->ws.modes, (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

extern "C" int32_t omk_pool_ensure_action(omk_ctx *c, const int32_t *ids, const int32_t *actions, int32_t n, int32_t evaluator) {
    CK(cudaSetDevice(c->device));
    int32_t rc = check_evaluator(c, evaluator);
    if (rc) return rc;
    if (!actions) return fail(OMK_ERR_INVALID, "actions is NULL");
    const int32_t *d_ids;
    rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    rc = ensure_workspace(c, n);
    if (rc) return rc;
    CK(copy_h2d(c, c->ws.actions, actions, sizeof(int32_t) * (size_t)n, c->stream));
    launch_reset_requests(c);
    launch_ensure_prepare(c, d_ids, c->ws.actions, n);
    RUN_EVAL(c, evaluator, n);
    launch_apply(c, d_ids, n, kApplyEnsure);
    return check_device_error(c);
}

extern "C" int32_t omk_pool_play(omk_ctx *c, const int32_t *ids, const int32_t *actions, int32_t n, int8_t *out_status) {
    CK(cudaSetDevice(c->device));
    if (!actions) return fail(OMK_ERR_INVALID, "actions is NULL");
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    CK(copy_h2d(c, c->ws.actions, actions, sizeof(int32_t) * (size_t)n, c->stream));
    launch_play(c, d_ids, c->ws.actions, n, c->ws.status);
    if (out_status) CK(copy_d2h(c, out_status, c->ws.status, (size_t)n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

struct RootDump {
    int32_t actions[kCells];
    unsigned long long n[kCells];
    float w[kCells], p[kCells];
    int32_t len;
    float policy[kCells];
    uint32_t misc[16];
};

static int32_t dump_root(omk_ctx *c, int32_t id, RootDump *host) {
    CK(cudaSetDevice(c->device));
    if (id < 0 || id >= c->cap_trees) return fail(OMK_ERR_INVALID, "tree id out of range");
    RootDump *d = nullptr;
    SCRATCH(0, 1, d);
    launch_root_children(c, id, d->actions, d->n, d->w, d->p, &d->len, d->policy, d->misc);
    CK(copy_d2h(c, host, d, sizeof(RootDump), c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

extern "C" int32_t omk_pool_root_children(omk_ctx *c, int32_t id, int32_t *out_actions, uint64_t *out_n, float *out_w,
                                          float *out_p, int32_t *out_len) {
    RootDump h;
    int32_t rc = dump_root(c, id, &h);
    if (rc) return rc;
    for (int i = 0; i < h.len; ++i) {
        if (out_actions) out_actions[i] = h.actions[i];
        if (out_n) out_n[i] = h.n[i];
        if (out_w) out_w[i] = h.w[i];
        if (out_p) out_p[i] = h.p[i];
    }
    if (out_len) *out_len = h.len;
    return OMK_OK;
}

extern "C" int32_t omk_pool_root_stats(omk_ctx *c, int32_t id, uint64_t *out_n, float *out_w, float *out_p, int32_t *out_status,
                                       float *out_policy) {
    RootDump h;
    int32_t rc = dump_root(c, id, &h);
    if (rc) return rc;
    if (out_n) *out_n = h.misc[0];
    if (out_w) memcpy(out_w, &h.misc[1], 4);
    if (out_p) memcpy(out_p, &h.misc[2], 4);
    if (out_status) *out_status = (int32_t)h.misc[3];
    if (out_policy) memcpy(out_policy, h.policy, sizeof h.policy);
    return OMK_OK;
}

extern "C" int32_t omk_pool_tree_info(omk_ctx *c, int32_t id, int32_t *out_nodes, uint32_t *out_rng_counter) {
    RootDump h;
    int32_t rc = dump_root(c, id, &h);
    if (rc) return rc;
    if (out_nodes) *out_nodes = (int32_t)h.misc[4];
    if (out_rng_counter) *out_rng_counter = h.misc[5];
    return OMK_OK;
}

extern "C" int32_t omk_pool_get_env(omk_ctx *c, int32_t id, uint8_t *out_board, uint8_t *out_turn, uint16_t *out_legal_count) {
    RootDump h;
    int32_t rc = dump_root(c, id, &h);
    if (rc) return rc;
    if (out_board)
        for (int i = 0; i < kCells; ++i) {
            const bool b = (h.misc[8 + (i >> 5)] >> (i & 31)) & 1u, w = (h.misc[11 + (i >> 5)] >> (i & 31)) & 1u;
            out_board[i] = b ? 1 : (w ? 2 : 0);
        }
    if (out_turn) *out_turn = (uint8_t)(h.misc[6] & 0xFF);
    if (out_legal_count) *out_legal_count = (uint16_t)((h.misc[6] >> 8) & 0xFF);
    return OMK_OK;
}

extern "C" int32_t omk_pool_get_envs(omk_ctx *c, const int32_t *ids, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                                     uint16_t *out_legal_counts, int8_t *out_status) {
    CK(cudaSetDevice(c->device));
    const int32_t *d_ids;
    int32_t rc = stage_ids(c, ids, n, &d_ids, c->cap_trees);
    if (rc) return rc;
    if (n == 0) return OMK_OK;
    // one scratch block: [boards n*81 | turns n | status n | legal n u16]
    uint8_t *blk = nullptr;
    const size_t nn = (size_t)n, off_t = nn * kCells, off_s = off_t + nn, off_l = (off_s + nn + 1) & ~(size_t)1;
    SCRATCH(0, off_l + 2 * nn, blk);
    launch_pool_get_envs(c, d_ids, n, blk, blk + off_t, reinterpret_cast<uint16_t *>(blk + off_l), reinterpret_cast<int8_t *>(blk + off_s));
    if (out_boards) CK(copy_d2h(c, out_boards, blk, nn * kCells, c->stream));
    if (out_turns) CK(copy_d2h(c, out_turns, blk + off_t, nn, c->stream));
    if (out_status) CK(copy_d2h(c, out_status, blk + off_s, nn, c->stream));
    if (out_legal_counts) CK(copy_d2h(c, out_legal_counts, blk + off_l, 2 * nn, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

// ------------------------------------------------------------------ self-play driver
struct SpLayout {
    int32_t *mover, *other, *actions;
    float *temps;
    uint8_t *modes;
    int8_t *status, *status2;
    float *root_policy;
    unsigned long long *counters;  // [0] games finished
    size_t bytes;
};
// one ply slot of the transition ring: [boards n*81 u8 | policy n*81 f32 | actions n i32 | status n i8], 256-byte aligned parts
struct SpSlot {
    size_t off_boards, off_policy, off_actions, off_status, bytes;
};
static SpSlot sp_slot_layout(int n) {
    SpSlot s;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    s.off_boards = 0;
    s.off_policy = up((size_t)n * kCells);
    s.off_actions = s.off_policy + up((size_t)n * kCells * sizeof(float));
    s.off_status = s.off_actions + up((size_t)n * sizeof(int32_t));
    s.bytes = s.off_status + up((size_t)n);
    return s;
}
static SpLayout sp_layout(uint8_t *base, int n) {
    SpLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t *p = base + off; off = (off + bytes + 255) & ~(size_t)255; return p; };
    L.mover = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * (size_t)n));
    L.other = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * (size_t)n));
    L.actions = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * (size_t)n));
    L.temps = reinterpret_cast<float *>(take(sizeof(float) * (size_t)n));
    L.modes = take((size_t)n);
    L.status = reinterpret_cast<int8_t *>(take((size_t)n));
    L.status2 = reinterpret_cast<int8_t *>(take((size_t)n));
    L.root_policy = reinterpret_cast<float *>(take(sizeof(float) * kRow));
    L.counters = reinterpret_cast<unsigned long long *>(take(64));
    L.bytes = off;
    return L;
}
// Restarted games install a cached raw prior of the empty board instead of evaluating it again (Agent::new, agent.rs:16-25,
// evaluates with the CURRENT weights).  The cache therefore follows every weight change: omk_net_load_params and
// omk_net_init_random call this while a self-play driver is active (trainer step -> sync weights -> next self-play phase).
static int32_t sp_refresh_root_policy(omk_ctx *c) {
    if (!c->sp_active || c->sp_cfg.evaluator != OMK_EVAL_NET) return OMK_OK;
    int32_t rc = ensure_workspace(c, 1);
    if (rc) return rc;
    const SpLayout L = sp_layout(c->sp_buf, c->sp_cfg.n_games);
    const uint32_t one = 1;
    CK(cudaMemsetAsync(c->ws.nn_in, 0, sizeof(NNIn), c->stream));  // empty board, Black to move, EnvTurnMode::Player (== k_new_games' request)
    CK(copy_h2d(c, c->ws.n_req, &one, sizeof one, c->stream));
    if (!net_forward(c, nullptr, 1)) return fail(OMK_ERR_CUDA, "re-evaluating the empty board after a weight change failed");
    CK(cudaMemcpyAsync(L.root_policy, c->ws.P, sizeof(float) * kCells, cudaMemcpyDeviceToDevice, c->stream));
    launch_reset_requests(c);
    return check_device_error(c);
}

extern "C" int32_t omk_selfplay_begin(omk_ctx *c, const omk_selfplay_config *cfg) {
    CK(cudaSetDevice(c->device));
    if (!cfg) return fail(OMK_ERR_INVALID, "cfg is NULL");
    if (cfg->n_games < 1 || 2 * cfg->n_games > c->cap_trees) return fail(OMK_ERR_INVALID, "need capacity_trees >= 2*n_games");
    if (cfg->batch_size < 1 || cfg->batch_size > kMaxBatchPerTree || cfg->count < 1) return fail(OMK_ERR_INVALID, "bad count/batch_size");
    int32_t rc = check_evaluator(c, cfg->evaluator);
    if (rc) return rc;
    const int n = cfg->n_games;
    const int rows = n * cfg->batch_size > 2 * n ? n * cfg->batch_size : 2 * n;
    rc = ensure_workspace(c, rows);
    if (rc) return rc;
    // The driver's buffers are allocated into locals and committed together below: a failed allocation leaves no driver
    // (sp_active false) rather than half of one.  Each old buffer is released before its successor is allocated.
    c->sp_active = false;
    c->sp_cfg = *cfg;
    const SpSlot slot = sp_slot_layout(n);
    const bool new_ring = slot.bytes != c->sp_ring_slot_bytes;
    c->sp_ply.reset();
    c->sp_buf.reset();
    Buf<int32_t> ply;
    Buf<uint8_t> buf, ring_dev;
    PinnedBuf<uint8_t> ring_host;
    CK(ply.alloc((size_t)n));
    CK(cudaMemsetAsync(ply, 0, ply.bytes(), c->stream));
    CK(buf.alloc(sp_layout(nullptr, n).bytes));
    CK(cudaMemsetAsync(buf, 0, buf.bytes(), c->stream));
    // transition ring: device slots + pinned host mirror + copy stream + events
    if (new_ring) {
        c->sp_ring_dev.reset();
        c->sp_ring_host.reset();
        c->sp_ring_slot_bytes = 0;
        CK(ring_dev.alloc(slot.bytes * omk_ctx::kSpRing));
        CK(ring_host.alloc(slot.bytes * omk_ctx::kSpRing));
    }
    if (!c->sp_copy_stream) {
        CK(cudaStreamCreateWithFlags(&c->sp_copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < omk_ctx::kSpRing; ++i) {
            CK(cudaEventCreateWithFlags(&c->sp_ev_rec[i][0], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&c->sp_ev_rec[i][1], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&c->sp_ev_copy[i], cudaEventDisableTiming));
        }
    }
    // a replay memory that exists now is fed by this driver: staging for every game (the restart below drops the tails
    // of the previous driver's games, as omk_selfplay_begin restarts every game)
    Replay &r = c->rp;
    if (r.stream) cudaStreamSynchronize(r.stream);  // the last commit reads the old staging
    r.stage = ReplayStaging{};
    ReplayStaging stage;
    if (r.ring.cap > 0) {
        if (!r.stream) {
            CK(cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&r.ev_commit, cudaEventDisableTiming));
        }
        const size_t cells = (size_t)n * kCells * kCells;  // 81 plies of 81 cells per game
        CK(stage.boards.alloc(cells));
        CK(stage.pi.alloc(cells));
        CK(stage.len.alloc((size_t)n));
        CK(cudaMemsetAsync(stage.len, 0, stage.len.bytes(), c->stream));
        stage.games = n;
    }
    c->sp_ply = std::move(ply);
    c->sp_buf = std::move(buf);
    if (new_ring) {
        c->sp_ring_dev = std::move(ring_dev);
        c->sp_ring_host = std::move(ring_host);
        c->sp_ring_slot_bytes = slot.bytes;
    }
    r.stage = std::move(stage);
    const SpLayout M = sp_layout(c->sp_buf, n);
    // Agent::new for all 2n trees (stream id = tree id); then cache the root's raw policy for restarts:
    // evaluating the empty board is deterministic, so reusing it is bit-identical to evaluating it again
    launch_reset_requests(c);
    launch_new_games(c, nullptr, 2 * n, nullptr, nullptr, nullptr);
    RUN_EVAL(c, cfg->evaluator, 2 * n);
    launch_apply(c, nullptr, 2 * n, kApplyNewGame);
    CK(cudaMemcpyAsync(M.root_policy, c->tree_nodes + kOffPolicy, sizeof(float) * kCells, cudaMemcpyDeviceToDevice, c->stream));
    c->sp_active = true;
    return check_device_error(c);
}

extern "C" int32_t omk_selfplay_run(omk_ctx *c, int32_t plies, int32_t profile, uint8_t *out_boards, float *out_policy,
                                    int8_t *out_status, int32_t *out_actions, omk_selfplay_stats *stats) {
    CK(cudaSetDevice(c->device));
    if (!c->sp_active) return fail(OMK_ERR_STATE, "omk_selfplay_begin has not been called");
    if (plies < 0) return fail(OMK_ERR_INVALID, "plies < 0");
    if (c->sp_cfg.evaluator == OMK_EVAL_NET) {  // weights updated by the trainer since the last evaluation: operand images + the cached root prior
        int32_t rc_p = ensure_packed(c);
        if (rc_p) return rc_p;
    }
    const omk_selfplay_config &cfg = c->sp_cfg;
    const int n = cfg.n_games;
    const int rounds = (cfg.count + cfg.batch_size - 1) / cfg.batch_size;

    const SpLayout L = sp_layout(c->sp_buf, n);
    int32_t *mover = L.mover, *other = L.other, *actions = L.actions;
    float *temps = L.temps;
    uint8_t *modes = L.modes;
    int8_t *status = L.status, *status2 = L.status2;
    float *root_policy = L.root_policy;
    unsigned long long *counters = L.counters;

    // Transitions stream through a ring of kSpRing ply slots: the ply's kernels record into device slot ply % kSpRing, the
    // slice is copied to the pinned host mirror on the copy stream while later plies search, and the host drains a slot
    // into the caller's [ply][game] arrays just before the device reuses it (the host thread is then at most kSpRing
    // plies ahead of the GPU).
    constexpr int kRing = omk_ctx::kSpRing;
    const size_t tot = (size_t)plies * (size_t)n;
    const SpSlot slot = sp_slot_layout(n);
    const bool want_out = out_boards || out_policy || out_status || out_actions;
    // Replay feed (when a replay memory existed at omk_selfplay_begin): each lane stages its recorded ply per game; one
    // commit per ply on the replay stream, behind both lanes' record events, turns the episodes that ended into rows.  A
    // restarted game stages ply 0 over the finished episode, so each lane waits for the previous ply's commit before its
    // staging kernel -- one event wait per lane and ply, outside the search rounds.
    const bool feed = c->rp.stage.games == n && c->rp.ring.cap > 0;
    size_t d2h = 0;
    auto dev_slot = [&](int ply) { return c->sp_ring_dev + (size_t)(ply % kRing) * slot.bytes; };
    auto drain = [&](int ply) -> int32_t {  // pinned slot of `ply` -> the caller's arrays
        CK(cudaEventSynchronize(c->sp_ev_copy[ply % kRing]));
        const uint8_t *h = c->sp_ring_host + (size_t)(ply % kRing) * slot.bytes;
        const size_t row = (size_t)ply * n;
        if (out_boards) memcpy(out_boards + row * kCells, h + slot.off_boards, (size_t)n * kCells);
        if (out_policy) memcpy(out_policy + row * kCells, h + slot.off_policy, (size_t)n * kCells * sizeof(float));
        if (out_actions) memcpy(out_actions + row, h + slot.off_actions, (size_t)n * sizeof(int32_t));
        if (out_status) memcpy(out_status + row, h + slot.off_status, (size_t)n);
        return OMK_OK;
    };
    unsigned long long h_before[2] = {0, 0}, h_after[2] = {0, 0}, h_fin0 = 0, h_fin1 = 0;
    CK(copy_d2h(c, h_before, c->dev_sims, sizeof h_before, c->stream));
    CK(copy_d2h(c, &h_fin0, counters, sizeof h_fin0, c->stream));
    CK(cudaStreamSynchronize(c->stream));

    c->prof_level = profile;
    auto span_begin = [&](int kind) { return prof_begin(c, kind, 2); };
    auto span_end = [&](bool sp) { prof_end(c, sp); };

    // Two search lanes (halves of the games) when the pool is large enough: two independent kernel chains on two streams.
    const int lanes = lanes_for(c, n);
    const int lane_n[2] = {lanes == 2 ? (n + 1) / 2 : n, lanes == 2 ? n / 2 : 0};
    const int lane_g0[2] = {0, lane_n[0]};
    float *policy_out = c->ws.policy_out;
    for (int l = 0; l < lanes; ++l) {
        LaneScope scope(c, l, 0);
        int32_t rc_ws = ensure_workspace(c, lane_n[l] * cfg.batch_size);
        if (rc_ws) return rc_ws;
    }
    CK(cudaEventRecord(c->ev0, c->stream));
    if (lanes == 2) lanes_fork(c);
    for (int ply = 0; ply < plies; ++ply) {
        if (want_out && ply >= kRing) {  // the slot this ply records into still holds ply - kRing: hand it to the caller first
            int32_t rc_d = drain(ply - kRing);
            if (rc_d) return rc_d;
        }
        uint8_t *ds = dev_slot(ply);
        uint8_t *d_boards = ds + slot.off_boards;
        float *d_policy = reinterpret_cast<float *>(ds + slot.off_policy);
        int32_t *d_actions = reinterpret_cast<int32_t *>(ds + slot.off_actions);
        int8_t *d_status = reinterpret_cast<int8_t *>(ds + slot.off_status);
        for (int l = 0; l < lanes; ++l) {
            LaneScope scope(c, l, 0);
            const int g0 = lane_g0[l], nl = lane_n[l];
            bool sp = span_begin(OMK_K_MOVE);
            launch_sp_prepare(c, g0, nl, mover, other, modes, temps);
            launch_root_noise(c, mover + g0, nl, cfg.epsilon, cfg.alpha);
            span_end(sp);
        }
        for (int r = 0; r < rounds; ++r) {
            for (int l = 0; l < lanes; ++l) {
                LaneScope scope(c, l, 0);
                const int g0 = lane_g0[l], nl = lane_n[l];
                bool sp = span_begin(OMK_K_SELECT);
                launch_reset_requests(c);
                launch_select_expand(c, mover + g0, nl, cfg.batch_size);
                span_end(sp);
                RUN_EVAL(c, cfg.evaluator, nl * cfg.batch_size);
                sp = span_begin(OMK_K_APPLY);
                launch_apply(c, mover + g0, nl, kApplySearch);
                span_end(sp);
            }
        }
        for (int l = 0; l < lanes; ++l) {
            LaneScope scope(c, l, 0);
            const int g0 = lane_g0[l], nl = lane_n[l];
            const size_t row = (size_t)g0;  // within the ply's ring slot
            bool sp = span_begin(OMK_K_MOVE);
            launch_sample(c, mover + g0, nl, modes + g0, temps + g0, actions + g0, policy_out + (size_t)g0 * kCells, nullptr);
            launch_sp_record(c, nl, mover + g0, actions + g0, policy_out + (size_t)g0 * kCells, d_boards + row * kCells,
                             d_policy + row * kCells, d_actions + row);
            if (feed) {
                CK(cudaStreamWaitEvent(c->stream, c->rp.ev_commit, 0));
                launch_rp_stage(c, g0, nl, d_boards + row * kCells, d_policy + row * kCells);
            }
            launch_play(c, mover + g0, actions + g0, nl, status + g0);
            launch_reset_requests(c);
            launch_ensure_prepare(c, other + g0, actions + g0, nl);
            span_end(sp);
            RUN_EVAL(c, cfg.evaluator, nl);
            sp = span_begin(OMK_K_MOVE);
            launch_apply(c, other + g0, nl, kApplyEnsure);
            launch_play(c, other + g0, actions + g0, nl, status2 + g0);
            CK(cudaMemcpyAsync(d_status + row, status + g0, (size_t)nl, cudaMemcpyDeviceToDevice, c->stream));
            // finished games restart with fresh trees for both colours (cached root policy) and ply 0
            launch_new_games(c, mover + g0, nl, nullptr, status + g0, root_policy);
            launch_new_games(c, other + g0, nl, nullptr, status + g0, root_policy);
            launch_sp_advance(c, g0, nl, status, counters);
            span_end(sp);
            if (want_out || feed) CK(cudaEventRecord(c->sp_ev_rec[ply % kRing][l], c->stream));
        }
        if (feed) {  // this ply's finished episodes -> replay rows, behind both lanes' status of the ply
            for (int l = 0; l < lanes; ++l) CK(cudaStreamWaitEvent(c->rp.stream, c->sp_ev_rec[ply % kRing][l], 0));
            launch_rp_commit(c, n, d_status);
            CK(cudaEventRecord(c->rp.ev_commit, c->rp.stream));
        }
        if (want_out) {  // this ply's slice -> pinned host mirror, behind both lanes' recording kernels
            for (int l = 0; l < lanes; ++l) CK(cudaStreamWaitEvent(c->sp_copy_stream, c->sp_ev_rec[ply % kRing][l], 0));
            uint8_t *hs = c->sp_ring_host + (size_t)(ply % kRing) * slot.bytes;
            if (out_boards) { CK(copy_d2h(c, hs + slot.off_boards, d_boards, (size_t)n * kCells, c->sp_copy_stream)); d2h += (size_t)n * kCells; }
            if (out_policy) { CK(copy_d2h(c, hs + slot.off_policy, d_policy, (size_t)n * kCells * sizeof(float), c->sp_copy_stream)); d2h += (size_t)n * kCells * 4; }
            if (out_actions) { CK(copy_d2h(c, hs + slot.off_actions, d_actions, (size_t)n * 4, c->sp_copy_stream)); d2h += (size_t)n * 4; }
            if (out_status) { CK(copy_d2h(c, hs + slot.off_status, d_status, (size_t)n, c->sp_copy_stream)); d2h += (size_t)n; }
            CK(cudaEventRecord(c->sp_ev_copy[ply % kRing], c->sp_copy_stream));
            // the device slot is recorded into again kRing plies from now: by then the host has waited for this copy (drain)
        }
    }
    if (lanes == 2) {
        LaneScope scope(c, 1, 0);
        launch_reset_requests(c);
    }
    if (lanes == 2) lanes_join(c);
    launch_reset_requests(c);  // folds the last round's request count into the evaluator total
    if (feed) CK(cudaStreamWaitEvent(c->stream, c->rp.ev_commit, 0));  // every later reader of the replay is behind the last commit
    CK(cudaEventRecord(c->ev1, c->stream));
    if (want_out)
        for (int ply = plies > kRing ? plies - kRing : 0; ply < plies; ++ply) {  // the slots still in flight
            int32_t rc_d = drain(ply);
            if (rc_d) return rc_d;
        }
    CK(copy_d2h(c, h_after, c->dev_sims, sizeof h_after, c->stream));
    CK(copy_d2h(c, &h_fin1, counters, sizeof h_fin1, c->stream));
    ReplayCounters rp_ctr{};
    if (feed) CK(copy_d2h(c, &rp_ctr, c->rp.counters, sizeof rp_ctr, c->stream));
    int32_t rc = check_device_error(c);  // (synchronises the stream)
    if (feed) {
        c->rp.added = rp_ctr.added;
        c->rp.len = rp_ctr.len;
        c->rp.episodes = rp_ctr.episodes;
    }
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->simulations = (int64_t)(h_after[0] - h_before[0]);
        stats->nn_evals = (int64_t)(h_after[1] - h_before[1]);
        stats->positions = (int64_t)tot;
        stats->games_finished = (int64_t)(h_fin1 - h_fin0);
        stats->d2h_bytes = (int64_t)d2h;
        stats->h2d_bytes = 0;
        cudaEventElapsedTime(&stats->gpu_ms, c->ev0, c->ev1);
        for (auto &s : c->prof_spans) {
            float ms = 0;
            cudaEventElapsedTime(&ms, s.a, s.b);
            stats->kind_ms[s.kind] += ms;
            stats->kind_launches[s.kind] += 1;
        }
    }
    for (auto &s : c->prof_spans) {
        c->prof_pool.push_back(s.a);
        c->prof_pool.push_back(s.b);
    }
    c->prof_spans.clear();
    c->prof_level = 0;
    return rc;
}

// ------------------------------------------------------------------ replay memory (src/trainer.rs:27,206-352 on the device)
extern "C" int32_t omk_replay_reset(omk_ctx *c, int64_t capacity) {
    CK(cudaSetDevice(c->device));
    if (capacity < 0 || capacity > 0x7FFFFFFFLL) return fail(OMK_ERR_INVALID, "capacity must be in [0, 2^31)");
    Replay &r = c->rp;
    if (capacity > 0 && r.ring.cap == 0 && c->sp_active)
        return fail(OMK_ERR_STATE, "a replay memory is fed by the self-play driver only if it exists at omk_selfplay_begin: create it first");
    CK(cudaStreamSynchronize(c->stream));
    if (capacity == 0) {  // the driver stops feeding
        if (r.stream) cudaStreamSynchronize(r.stream);
        r.stage = ReplayStaging{};
        r.ring = ReplayStore{};
        r.counters.reset();
        r.added = r.len = r.episodes = 0;
        return OMK_OK;
    }
    if (capacity != r.ring.cap) {
        if (r.stream) CK(cudaStreamSynchronize(r.stream));
        r.ring = ReplayStore{};
        const size_t cap = (size_t)capacity;
        ReplayStore ring;
        CK(ring.boards.alloc(cap * kCells));
        CK(ring.turns.alloc(cap));
        CK(ring.pi.alloc(cap * kCells));
        CK(ring.z.alloc(cap));
        ring.cap = capacity;
        r.ring = std::move(ring);
    }
    if (!r.counters) CK(r.counters.alloc(1));
    CK(cudaMemsetAsync(r.counters, 0, r.counters.bytes(), c->stream));  // the staged tails of a running driver stay
    CK(cudaStreamSynchronize(c->stream));
    r.added = r.len = r.episodes = 0;
    return OMK_OK;
}

extern "C" int32_t omk_replay_info(omk_ctx *c, int64_t *out_len, int64_t *out_rows_added, int64_t *out_episodes) {
    if (out_len) *out_len = c->rp.len;
    if (out_rows_added) *out_rows_added = c->rp.added;
    if (out_episodes) *out_episodes = c->rp.episodes;
    return OMK_OK;
}

// host row list -> device (validated against the current length)
static int32_t stage_rows(omk_ctx *c, const int64_t *rows, int32_t n, int64_t **out) {
    for (int32_t i = 0; i < n; ++i)
        if (rows[i] < 0 || rows[i] >= c->rp.len)
            return fail(OMK_ERR_INVALID, "row " + std::to_string(rows[i]) + " outside the replay's " + std::to_string(c->rp.len) + " rows");
    SCRATCH(0, (size_t)n, *out);
    CK(copy_h2d(c, *out, rows, sizeof(int64_t) * (size_t)n, c->stream));
    return OMK_OK;
}

extern "C" int32_t omk_replay_get(omk_ctx *c, const int64_t *rows, int32_t n, uint8_t *out_boards, uint8_t *out_turns,
                                  float *out_policy, float *out_z) {
    CK(cudaSetDevice(c->device));
    if (n < 0 || (n > 0 && !rows)) return fail(OMK_ERR_INVALID, "bad row list");
    if (c->rp.ring.cap == 0) return fail(OMK_ERR_STATE, "no replay memory (omk_replay_reset)");
    if (n == 0) return OMK_OK;
    int64_t *d_rows = nullptr;
    int32_t rc = stage_rows(c, rows, n, &d_rows);
    if (rc) return rc;
    const size_t nn = (size_t)n;
    uint8_t *d_bt = nullptr;  // [boards n*81 | turns n]
    float *d_pz = nullptr;    // [policy n*81 | z n]
    SCRATCH(1, nn * (kCells + 1), d_bt);
    SCRATCH(2, nn * (kCells + 1), d_pz);
    launch_rp_get(c, d_rows, n, d_bt, d_bt + nn * kCells, d_pz, d_pz + nn * kCells);
    if (out_boards) CK(copy_d2h(c, out_boards, d_bt, nn * kCells, c->stream));
    if (out_turns) CK(copy_d2h(c, out_turns, d_bt + nn * kCells, nn, c->stream));
    if (out_policy) CK(copy_d2h(c, out_policy, d_pz, sizeof(float) * nn * kCells, c->stream));
    if (out_z) CK(copy_d2h(c, out_z, d_pz + nn * kCells, sizeof(float) * nn, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

extern "C" int32_t omk_train_replay(omk_ctx *c, uint64_t seed, int64_t first_step, int32_t steps, int32_t n, float *out_losses,
                                    int64_t *out_rows) {
    CK(cudaSetDevice(c->device));
    if (steps < 1 || n < 1 || !out_losses) return fail(OMK_ERR_INVALID, "need steps >= 1, n >= 1 and out_losses");
    if (!c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    const Replay &r = c->rp;
    if (r.ring.cap == 0) return fail(OMK_ERR_STATE, "no replay memory (omk_replay_reset)");
    if (r.len == 0) return fail(OMK_ERR_STATE, "the replay memory is empty");
    const int m = (int)(r.len < n ? r.len : n);  // choose_multiple: min(n, len) rows
    float *img = nullptr, *pi = nullptr, *z = nullptr;
    if (const char *e = train_minibatch_buffers(c, m, &img, &pi, &z)) return fail(OMK_ERR_CUDA, std::string("omk_train_replay: ") + e);
    int64_t *d_rows = nullptr;
    float *d_losses = nullptr;
    SCRATCH(0, (size_t)steps * m, d_rows);
    SCRATCH(1, (size_t)steps * 3, d_losses);
    c->train_n = 0;
    launch_rp_sample(c, seed, first_step, steps, r.len, m, d_rows);
    for (int s = 0; s < steps; ++s) {  // omk_train_step's sequence, the minibatch encoded on the device
        launch_rp_gather(c, d_rows + (size_t)s * m, m, img, pi, z);
        if (const char *e = train_backward_resident(c, m)) return fail(OMK_ERR_CUDA, std::string("omk_train_replay: ") + e);
        if (const char *e = train_apply_step(c)) return fail(OMK_ERR_CUDA, std::string("omk_train_replay: ") + e);
        c->net_pack_dirty = true;
        if (const char *e = train_report_losses_device(c, m, d_losses + 3 * (size_t)s))
            return fail(OMK_ERR_CUDA, std::string("omk_train_replay: ") + e);
    }
    CK(copy_d2h(c, out_losses, d_losses, sizeof(float) * 3 * (size_t)steps, c->stream));
    if (out_rows) {  // [steps][n]: the m rows of each step, then -1
        CK(cudaMemcpy2DAsync(out_rows, sizeof(int64_t) * (size_t)n, d_rows, sizeof(int64_t) * (size_t)m, sizeof(int64_t) * (size_t)m,
                             (size_t)steps, cudaMemcpyDeviceToHost, c->stream));
        c->d2h_bytes += (int64_t)sizeof(int64_t) * steps * m;
    }
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    if (out_rows)
        for (int s = 0; s < steps; ++s)
            for (int k = m; k < n; ++k) out_rows[(size_t)s * n + k] = -1;
    for (int i = 0; i < 3 * steps; ++i)
        if (!(out_losses[i] == out_losses[i]) || out_losses[i] > 3.0e38f) return fail(OMK_ERR_NUMERIC, "the training loss is not finite");
    return OMK_OK;
}

// ------------------------------------------------------------------ evaluation against the naive player (src/trainer.rs:487-603)
extern "C" int32_t omk_naive_move(omk_ctx *c, const uint8_t *boards, const uint8_t *turns, int32_t n, uint64_t seed,
                                  const uint32_t *streams, int32_t *out_actions, uint8_t *out_forced) {
    CK(cudaSetDevice(c->device));
    if (n < 0 || (n > 0 && (!boards || !turns || !out_actions))) return fail(OMK_ERR_INVALID, "bad arguments");
    for (size_t i = 0; i < (size_t)n * kCells; ++i)
        if (boards[i] > 2) return fail(OMK_ERR_INVALID, "a cell is not 0 (Empty), 1 (Black) or 2 (White)");
    for (int32_t i = 0; i < n; ++i)
        if (turns[i] > 1) return fail(OMK_ERR_INVALID, "a turn is not 0 (Black) or 1 (White)");
    if (n == 0) return OMK_OK;
    const size_t nn = (size_t)n;
    uint8_t *d_pos = nullptr, *d_forced = nullptr;  // [boards n*81 | turns n]
    uint32_t *d_sa = nullptr;                       // [streams n | actions n]
    SCRATCH(0, nn * (kCells + 1), d_pos);
    SCRATCH(1, 2 * nn, d_sa);
    SCRATCH(2, nn, d_forced);
    int32_t *d_actions = reinterpret_cast<int32_t *>(d_sa + nn);
    CK(copy_h2d(c, d_pos, boards, nn * kCells, c->stream));
    CK(copy_h2d(c, d_pos + nn * kCells, turns, nn, c->stream));
    if (streams) CK(copy_h2d(c, d_sa, streams, sizeof(uint32_t) * nn, c->stream));
    launch_naive_move_boards(c, d_pos, d_pos + nn * kCells, streams ? d_sa : nullptr, n, mix64(seed ^ kNaiveKey), d_actions,
                             out_forced ? d_forced : nullptr);
    CK(copy_d2h(c, out_actions, d_actions, sizeof(int32_t) * nn, c->stream));
    if (out_forced) CK(copy_d2h(c, out_forced, d_forced, nn, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return OMK_OK;
}

// fold every lane's pending request count into the evaluated-positions total (dev_sims[1])
static void fold_requests(omk_ctx *c) {
    if (c->lane1_stream) {
        lanes_fork(c);
        {
            LaneScope scope(c, 1, 0);
            launch_reset_requests(c);
        }
        lanes_join(c);
    }
    launch_reset_requests(c);
}

extern "C" int32_t omk_eval_naive(omk_ctx *c, int32_t episodes, int32_t first_tree, int32_t count, int32_t batch_size, float epsilon,
                                  float alpha, int32_t evaluator, uint64_t seed, int32_t *out_result, int8_t *out_moves,
                                  int8_t *out_status, int64_t *out_stats, float *out_gpu_ms) {
    CK(cudaSetDevice(c->device));
    if (!out_result) return fail(OMK_ERR_INVALID, "out_result is NULL");
    if (episodes < 1 || first_tree < 0 || first_tree > c->cap_trees - episodes)
        return fail(OMK_ERR_INVALID, "need episodes >= 1 and the trees first_tree .. first_tree + episodes - 1 inside capacity_trees");
    if (batch_size < 1 || batch_size > kMaxBatchPerTree) return fail(OMK_ERR_INVALID, "batch_size must be in [1, 64]");
    if (count < 1) return fail(OMK_ERR_INVALID, "count < 1");
    if (c->sp_active && first_tree < 2 * c->sp_cfg.n_games)
        return fail(OMK_ERR_STATE, "the trees overlap the active self-play driver's trees 0 .. 2 * n_games - 1");
    int32_t rc = check_evaluator(c, evaluator);  // with the network: weights a training step changed are packed first
    if (rc) return rc;
    const int E = episodes;
    const size_t e = (size_t)E;
    // [simulations and evaluations before / after (4 u64) | counters (4 i32) | final status E | moves E*81] leave in one copy;
    // then the live tree ids, the half-move's actions, each game's ply and the half-move's statuses
    const size_t off_cnt = 32, off_fin = 48, off_moves = off_fin + e, out_bytes = off_moves + e * kCells;
    const size_t off_ids = (out_bytes + 255) & ~(size_t)255, off_act = off_ids + 4 * e, off_ply = off_act + 4 * e, off_st = off_ply + 4 * e;
    CK(c->eval_buf.grow(c->stream, off_st + e, 4096));
    rc = ensure_workspace(c, E);
    if (rc) return rc;
    uint8_t *base = c->eval_buf;
    unsigned long long *sims = reinterpret_cast<unsigned long long *>(base);
    int32_t *counters = reinterpret_cast<int32_t *>(base + off_cnt);
    int8_t *fin = reinterpret_cast<int8_t *>(base + off_fin), *moves = reinterpret_cast<int8_t *>(base + off_moves);
    int32_t *ids = reinterpret_cast<int32_t *>(base + off_ids), *actions = reinterpret_cast<int32_t *>(base + off_act);
    int32_t *ply = reinterpret_cast<int32_t *>(base + off_ply);
    int8_t *status = reinterpret_cast<int8_t *>(base + off_st);
    const uint64_t key = mix64(seed ^ kNaiveKey);

    fold_requests(c);  // counts earlier calls left pending are not this call's
    CK(cudaMemcpyAsync(sims, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev0, c->stream));
    launch_eval_init(c, E, first_tree, ids, ply, moves, fin, counters);
    // Agent::new for every game's tree (stream id = tree id)
    launch_reset_requests(c);
    launch_new_games(c, ids, E, nullptr, nullptr, nullptr);
    RUN_EVAL(c, evaluator, E);
    launch_apply(c, ids, E, kApplyNewGame);
    int64_t n_moves = 0, syncs = 0;
    int32_t n = E;
    for (int half = 0; n > 0 && half < kCells; ++half) {  // a game ends after at most 81 moves
        if (half % 2 == 0) {  // the naive player (Black), then ensure_action_exists + play_action in the model's tree
            launch_naive_move_trees(c, ids, n, first_tree, ply, key, actions);
            launch_reset_requests(c);
            launch_ensure_prepare(c, ids, actions, n);
            RUN_EVAL(c, evaluator, n);
            launch_apply(c, ids, n, kApplyEnsure);
        } else {  // the model (White): execute(count, batch_size, epsilon, alpha) + sample_action(Best)
            rc = search_rounds(c, ids, n, count, batch_size, epsilon, alpha, evaluator);
            if (rc) return rc;
            launch_sample(c, ids, n, nullptr, nullptr, actions, nullptr, nullptr);
        }
        launch_play(c, ids, actions, n, status);
        launch_eval_advance(c, ids, n, actions, status, first_tree, ply, moves, fin, counters);
        n_moves += n;
        // the half-move's one host round trip: the live count sizes the next launches
        CK(copy_d2h(c, &n, counters + 3, sizeof n, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        ++syncs;
    }
    fold_requests(c);
    CK(cudaMemcpyAsync(sims + 2, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev1, c->stream));
    std::vector<uint8_t> host(out_bytes);
    CK(copy_d2h(c, host.data(), base, out_bytes, c->stream));
    rc = check_device_error(c);  // (synchronises the stream)
    ++syncs;
    if (rc) return rc;
    const unsigned long long *h_sims = reinterpret_cast<const unsigned long long *>(host.data());
    const int32_t *h_cnt = reinterpret_cast<const int32_t *>(host.data() + off_cnt);
    for (int k = 0; k < 3; ++k) out_result[k] = h_cnt[k];
    if (out_status) memcpy(out_status, host.data() + off_fin, e);
    if (out_moves) memcpy(out_moves, host.data() + off_moves, e * kCells);
    if (out_stats) {
        out_stats[0] = (int64_t)(h_sims[2] - h_sims[0]);
        out_stats[1] = (int64_t)(h_sims[3] - h_sims[1]);
        out_stats[2] = n_moves;
        out_stats[3] = syncs;
    }
    if (out_gpu_ms) CK(cudaEventElapsedTime(out_gpu_ms, c->ev0, c->ev1));
    return OMK_OK;
}

// ------------------------------------------------------------------ model slots, the opponent network and the arena (benchmark/src/main.rs:14-108)
// slot s's fp32 tensors, allocated on first use (all or nothing)
static int32_t model_alloc(omk_ctx *c, int slot) {
    NetWeights &m = c->slot(slot);
    if (m.t[0]) return OMK_OK;
    NetWeights w;
    for (int i = 0; i < kNetTensors; ++i) CK(w.t[i].alloc((size_t)kLens[i]));
    CK(w.heads_w.alloc(512 * 128));
    CK(w.heads_b.alloc(128));
    m = std::move(w);
    return OMK_OK;
}
// after slot s's fp32 tensors changed: its packed heads and operand images (what omk_net_load_params does for the network)
static int32_t model_prepare(omk_ctx *c, int slot) {
    ModelScope scope(c, slot);
    const std::string who = slot == 1 ? std::string(" (opponent)") : " (model slot " + std::to_string(slot) + ")";
    net_pack_heads(c);
    if (!fc16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split fc weight preparation failed" + who);
    if (!tower16_prepare_weights(c)) return fail(OMK_ERR_CUDA, "fp16-split tower weight preparation failed" + who);
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    c->slot(slot).loaded = true;
    return OMK_OK;
}
static int32_t check_model_slot(int slot) {
    if (slot == 0) return fail(OMK_ERR_INVALID, "slot 0 is the network: omk_net_load_params and the trainer own it");
    if (slot < 1 || slot >= kModelSlots) return fail(OMK_ERR_INVALID, "model slot out of range [1, " + std::to_string(kModelSlots - 1) + "]");
    return OMK_OK;
}

extern "C" int32_t omk_model_load_params(omk_ctx *c, int32_t slot, const float *const *tensors, const int64_t *lens) {
    CK(cudaSetDevice(c->device));
    int32_t rc = check_model_slot(slot);
    if (rc) return rc;
    for (int i = 0; i < kNetTensors; ++i)
        if (!tensors[i] || lens[i] != kLens[i])
            return fail(OMK_ERR_INVALID, "tensor " + std::to_string(i) + ": expected " + std::to_string(kLens[i]) + " elements");
    rc = model_alloc(c, slot);
    if (rc) return rc;
    NetWeights &m = c->slot(slot);
    m.loaded = false;  // until the images below are built
    for (int i = 0; i < kNetTensors; ++i)
        CK(copy_h2d(c, m.t[i], tensors[i], sizeof(float) * (size_t)kLens[i], c->stream));
    return model_prepare(c, slot);
}

extern "C" int32_t omk_model_from_net(omk_ctx *c, int32_t slot) {
    CK(cudaSetDevice(c->device));
    int32_t rc = check_model_slot(slot);
    if (rc) return rc;
    if (!c->net.loaded) return fail(OMK_ERR_STATE, "network weights not loaded");
    rc = model_alloc(c, slot);
    if (rc) return rc;
    NetWeights &m = c->slot(slot);
    m.loaded = false;
    for (int i = 0; i < kNetTensors; ++i)
        CK(cudaMemcpyAsync(m.t[i], c->net.t[i], sizeof(float) * (size_t)kLens[i], cudaMemcpyDeviceToDevice, c->stream));
    return model_prepare(c, slot);
}

extern "C" int32_t omk_model_eval(omk_ctx *c, int32_t slot, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode,
                                  float *out_p, float *out_v) {
    if (slot < 0 || slot >= kModelSlots) return fail(OMK_ERR_INVALID, "model slot out of range [0, " + std::to_string(kModelSlots - 1) + "]");
    return eval_boards(c, slot, boards, turns, n, mode, out_p, out_v);
}

extern "C" int32_t omk_opponent_load_params(omk_ctx *c, const float *const *tensors, const int64_t *lens) {
    return omk_model_load_params(c, 1, tensors, lens);
}
extern "C" int32_t omk_opponent_from_net(omk_ctx *c) { return omk_model_from_net(c, 1); }
extern "C" int32_t omk_opponent_eval(omk_ctx *c, const uint8_t *boards, const uint8_t *turns, int32_t n, int32_t mode, float *out_p,
                                     float *out_v) {
    return omk_model_eval(c, 1, boards, turns, n, mode, out_p, out_v);
}

// stage s of one mover's half-move in omk_match, on the lane and with the model in use: 0 = ensure_action_exists + play_action of
// the other model's previous move in the mover's trees (none before the first half-move); 1 .. rounds = the search rounds;
// rounds + 1 = sample_action(Best) + play_action
static int32_t match_stage(omk_ctx *c, int stage, int rounds, int half, const int32_t *trees, int n, int32_t *act, int8_t *status,
                           int8_t *other_status, int batch_size, float epsilon, float alpha, int evaluator) {
    if (stage == 0) {
        if (half == 0) return OMK_OK;
        launch_reset_requests(c);
        launch_ensure_prepare(c, trees, act, n);
        RUN_EVAL(c, evaluator, n);
        launch_apply(c, trees, n, kApplyEnsure);
        launch_play(c, trees, act, n, other_status);
        return OMK_OK;
    }
    if (stage <= rounds) return search_round(c, trees, n, stage - 1, batch_size, epsilon, alpha, evaluator);
    launch_sample(c, trees, n, nullptr, nullptr, act, nullptr, nullptr);
    launch_play(c, trees, act, n, status);
    return OMK_OK;
}

extern "C" int32_t omk_match(omk_ctx *c, int32_t pairs, int32_t first_tree, int32_t count, int32_t batch_size, float epsilon,
                             float alpha, int32_t evaluator, int32_t *out_result, int8_t *out_moves, int8_t *out_status,
                             int64_t *out_stats, float *out_gpu_ms) {
    CK(cudaSetDevice(c->device));
    if (!out_result) return fail(OMK_ERR_INVALID, "out_result is NULL");
    if (pairs < 1 || first_tree < 0 || (int64_t)first_tree + 4 * (int64_t)pairs > c->cap_trees)
        return fail(OMK_ERR_INVALID, "need pairs >= 1 and the trees first_tree .. first_tree + 4 * pairs - 1 inside capacity_trees");
    if (batch_size < 1 || batch_size > kMaxBatchPerTree) return fail(OMK_ERR_INVALID, "batch_size must be in [1, 64]");
    if (count < 1) return fail(OMK_ERR_INVALID, "count < 1");
    if (evaluator != OMK_EVAL_NET && evaluator != OMK_EVAL_HASH) return fail(OMK_ERR_INVALID, "unknown evaluator");
    if (c->sp_active && first_tree < 2 * c->sp_cfg.n_games)
        return fail(OMK_ERR_STATE, "the trees overlap the active self-play driver's trees 0 .. 2 * n_games - 1");
    int32_t rc = check_evaluator(c, evaluator);  // with the network: weights a training step changed are packed first
    if (rc) return rc;
    if (evaluator == OMK_EVAL_NET && !c->opp.loaded)
        return fail(OMK_ERR_STATE, "opponent weights not loaded (omk_opponent_load_params / omk_opponent_from_net)");
    const int P = pairs;
    const size_t g = 2 * (size_t)P;  // games
    // [simulations and evaluations before / after (4 u64) | counters (8 i32) | final status g | moves g*81] leave in one copy;
    // then the tree ids [model][leg][P] (network 0, opponent 1), the games' random streams [g], and per leg [leg][P] the moves
    // of the half-move, the mover's statuses and the statuses of the other model's play_action
    const size_t off_cnt = 32, off_fin = 64, off_moves = off_fin + g, out_bytes = off_moves + g * kCells;
    const size_t off_ids = (out_bytes + 255) & ~(size_t)255, off_str = off_ids + 8 * g, off_act = off_str + 4 * g, off_st = off_act + 4 * g,
                 off_ost = off_st + g;
    CK(c->eval_buf.grow(c->stream, off_ost + g, 4096));
    // both legs run at once, the network's half-move on lane 0 and the opponent's on lane 1
    const bool two_lanes = c->lane_min_trees > 0 && lane1_ready(c);
    const int rows = P * batch_size > 2 * P ? P * batch_size : 2 * P;
    for (int l = 0; l < (two_lanes ? 2 : 1); ++l) {
        LaneScope scope(c, l, 0);
        rc = ensure_workspace(c, rows);
        if (rc) return rc;
    }
    uint8_t *base = c->eval_buf;
    unsigned long long *sims = reinterpret_cast<unsigned long long *>(base);
    int32_t *counters = reinterpret_cast<int32_t *>(base + off_cnt);
    int8_t *fin = reinterpret_cast<int8_t *>(base + off_fin), *moves = reinterpret_cast<int8_t *>(base + off_moves);
    int32_t *ids = reinterpret_cast<int32_t *>(base + off_ids), *actions = reinterpret_cast<int32_t *>(base + off_act);
    uint32_t *streams = reinterpret_cast<uint32_t *>(base + off_str);
    int8_t *status = reinterpret_cast<int8_t *>(base + off_st), *other_status = reinterpret_cast<int8_t *>(base + off_ost);

    fold_requests(c);  // counts earlier calls left pending are not this call's
    CK(cudaMemcpyAsync(sims, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev0, c->stream));
    launch_match_init(c, P, first_tree, ids, streams, moves, fin, counters);
    for (int m = 0; m < 2; ++m) {  // Agent::new for every game's tree of model m, under model m's weights
        ModelScope scope(c, m == 1);
        launch_reset_requests(c);
        launch_new_games(c, ids + m * g, (int)g, streams, nullptr, nullptr);
        RUN_EVAL(c, evaluator, (int)g);
        launch_apply(c, ids + m * g, (int)g, kApplyNewGame);
    }
    const int rounds = (count + batch_size - 1) / batch_size;  // parallel_mcts_executor.rs:39-42,207
    int32_t back[3] = {0, P, P};  // {device error word, live games in leg 0, in leg 1}
    int *live = back + 1;
    int64_t n_moves = 0, syncs = 0;
    // a game ends after at most 81 moves; a device error (out of node slots, a non-finite network output, a refused move)
    // ends the match at the half-move that raised it
    for (int half = 0; (live[0] > 0 || live[1] > 0) && back[0] == 0 && half < kCells; ++half) {
        // the movers of this half-move: the network in leg half % 2, the opponent in the other leg
        struct Part {
            int leg;
            bool opponent;
        } part[2];
        int parts = 0;
        for (int m = 0; m < 2; ++m) {
            const int leg = (half + m) % 2;
            if (live[leg] > 0) part[parts++] = {leg, m == 1};
        }
        const int lanes = two_lanes && parts == 2 ? 2 : 1;
        if (lanes == 2) lanes_fork(c);
        for (int stage = 0; stage < rounds + 2 && rc == OMK_OK; ++stage)
            for (int p = 0; p < parts && rc == OMK_OK; ++p) {
                LaneScope lane(c, lanes == 2 ? p : 0, 0);
                ModelScope model(c, part[p].opponent);
                const int leg = part[p].leg;
                rc = match_stage(c, stage, rounds, half, ids + ((part[p].opponent ? 2 : 0) + leg) * P, live[leg], actions + leg * P,
                                 status + leg * P, other_status + leg * P, batch_size, epsilon, alpha, evaluator);
            }
        if (lanes == 2) lanes_join(c);  // on an error too: nothing queued on lane 1 is left unordered with the main stream
        if (rc) return rc;
        launch_match_advance(c, P, first_tree, half, live, ids, actions, status, other_status, moves, fin, counters);
        n_moves += live[0] + live[1];
        // the half-move's one host round trip: both legs' live counts size the next launches
        CK(copy_d2h(c, back, counters + 3, sizeof back, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        ++syncs;
    }
    fold_requests(c);
    CK(cudaMemcpyAsync(sims + 2, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev1, c->stream));
    std::vector<uint8_t> host(out_bytes);
    CK(copy_d2h(c, host.data(), base, out_bytes, c->stream));
    rc = check_device_error(c);  // (synchronises the stream)
    ++syncs;
    if (rc) return rc;
    const unsigned long long *h_sims = reinterpret_cast<const unsigned long long *>(host.data());
    const int32_t *h_cnt = reinterpret_cast<const int32_t *>(host.data() + off_cnt);
    for (int k = 0; k < 3; ++k) out_result[k] = h_cnt[k];
    if (out_status) memcpy(out_status, host.data() + off_fin, g);
    if (out_moves) memcpy(out_moves, host.data() + off_moves, g * kCells);
    if (out_stats) {
        out_stats[0] = (int64_t)(h_sims[2] - h_sims[0]);
        out_stats[1] = (int64_t)(h_sims[3] - h_sims[1]);
        out_stats[2] = n_moves;
        out_stats[3] = syncs;
    }
    if (out_gpu_ms) CK(cudaEventElapsedTime(out_gpu_ms, c->ev0, c->ev1));
    return OMK_OK;
}

// ------------------------------------------------------------------ the tournament: omk_match over every pairing of up to 16 models
// naive: participant 0 is the naive player (seeded by `seed`, DESIGN.md 4) and participant k + 1 is slots[k]; otherwise
// participant k is slots[k] and `seed` is unused
static int32_t tournament(omk_ctx *c, bool naive, int32_t n_models, const int32_t *slots, int32_t pairs, int32_t first_tree, int32_t count,
                          int32_t batch_size, float epsilon, float alpha, int32_t evaluator, uint64_t seed, int32_t *out_result,
                          int8_t *out_moves, int8_t *out_status, int64_t *out_stats, float *out_gpu_ms) {
    CK(cudaSetDevice(c->device));
    if (!out_result) return fail(OMK_ERR_INVALID, "out_result is NULL");
    const int min_models = naive ? 1 : 2;
    if (n_models < min_models || n_models > kModelSlots || !slots)
        return fail(OMK_ERR_INVALID, "need " + std::to_string(min_models) + " <= n_models <= " + std::to_string(kModelSlots) + " and a slot list");
    bool listed[kModelSlots] = {};
    for (int m = 0; m < n_models; ++m) {
        if (slots[m] < 0 || slots[m] >= kModelSlots) return fail(OMK_ERR_INVALID, "model slot out of range [0, " + std::to_string(kModelSlots - 1) + "]");
        if (listed[slots[m]]) return fail(OMK_ERR_INVALID, "duplicate model slot in the tournament");
        listed[slots[m]] = true;
    }
    const int n = n_models + (naive ? 1 : 0), P = n * (n - 1) / 2;  // participants, pairings
    const int first_model = naive ? 1 : 0;
    auto slot_of = [&](int m) { return slots[m - first_model]; };  // participant m >= first_model
    if (pairs < 1 || first_tree < 0 || (int64_t)first_tree + 4 * (int64_t)pairs * P > c->cap_trees)
        return fail(OMK_ERR_INVALID, "need pairs >= 1 and the trees first_tree .. first_tree + 4 * pairs * n(n-1)/2 - 1 inside capacity_trees");
    if (batch_size < 1 || batch_size > kMaxBatchPerTree) return fail(OMK_ERR_INVALID, "batch_size must be in [1, 64]");
    if (count < 1) return fail(OMK_ERR_INVALID, "count < 1");
    if (evaluator != OMK_EVAL_NET && evaluator != OMK_EVAL_HASH) return fail(OMK_ERR_INVALID, "unknown evaluator");
    if (c->sp_active && first_tree < 2 * c->sp_cfg.n_games)
        return fail(OMK_ERR_STATE, "the trees overlap the active self-play driver's trees 0 .. 2 * n_games - 1");
    int32_t rc = check_evaluator(c, evaluator);  // with the network: weights a training step changed are packed first
    if (rc) return rc;
    if (evaluator == OMK_EVAL_NET)
        for (int m = 0; m < n_models; ++m)
            if (!c->slot(slots[m]).loaded) return fail(OMK_ERR_STATE, slot_name(slots[m]) + " weights not loaded");
    const int Q = pairs;
    const size_t G = 2 * (size_t)Q * P;  // games
    const int gcap = (n - 1) * 2 * Q;     // a participant's trees: its init list, and twice its largest group
    // [simulations and evaluations before / after (4 u64) | counters [P][3] i32 | final status G | moves G*81] leave in one copy;
    // then the per-pairing lists and the per-model groups (TourneyState)
    const size_t off_cnt = 32, off_fin = off_cnt + 12 * (size_t)P, off_moves = off_fin + G, out_bytes = off_moves + G * kCells;
    size_t end = (out_bytes + 255) & ~(size_t)255;
    auto take = [&](size_t bytes) {
        const size_t o = end;
        end = (end + bytes + 15) & ~(size_t)15;
        return o;
    };
    const size_t mg = (size_t)n * gcap;
    const size_t off_ids = take(8 * G), off_act = take(4 * G), off_live = take(8 * (size_t)P), off_off = take(8 * (size_t)P),
                 off_back = take(4 * (size_t)(n + 1)), off_gids = take(4 * mg), off_gact = take(4 * mg), off_gstr = take(4 * mg),
                 off_gst = take(mg), off_gost = take(mg);
    CK(c->eval_buf.grow(c->stream, end, 4096));
    // the groups run interleaved over both lanes, group k on lane k % 2
    const bool two_lanes = c->lane_min_trees > 0 && lane1_ready(c);
    const int rows = (n - 1) * Q * batch_size > gcap ? (n - 1) * Q * batch_size : gcap;
    for (int l = 0; l < (two_lanes ? 2 : 1); ++l) {
        LaneScope scope(c, l, 0);
        rc = ensure_workspace(c, rows);
        if (rc) return rc;
    }
    uint8_t *base = c->eval_buf;
    unsigned long long *sims = reinterpret_cast<unsigned long long *>(base);
    TourneyState t;
    t.n = n;
    t.pairs = Q;
    t.first_tree = first_tree;
    t.gcap = gcap;
    t.naive = naive ? 1 : 0;
    t.counters = reinterpret_cast<int32_t *>(base + off_cnt);
    t.final_status = reinterpret_cast<int8_t *>(base + off_fin);
    t.moves = reinterpret_cast<int8_t *>(base + off_moves);
    t.ids = reinterpret_cast<int32_t *>(base + off_ids);
    t.actions = reinterpret_cast<int32_t *>(base + off_act);
    t.live = reinterpret_cast<int32_t *>(base + off_live);
    t.off = reinterpret_cast<int32_t *>(base + off_off);
    t.back = reinterpret_cast<int32_t *>(base + off_back);
    t.gids = reinterpret_cast<int32_t *>(base + off_gids);
    t.gact = reinterpret_cast<int32_t *>(base + off_gact);
    t.gstr = reinterpret_cast<uint32_t *>(base + off_gstr);
    t.gst = reinterpret_cast<int8_t *>(base + off_gst);
    t.gost = reinterpret_cast<int8_t *>(base + off_gost);

    fold_requests(c);  // counts earlier calls left pending are not this call's
    CK(cudaMemcpyAsync(sims, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev0, c->stream));
    launch_tourney_init(c, t);
    for (int m = first_model; m < n; ++m) {  // Agent::new for every tree of model m, under model m's weights
        ModelScope scope(c, slot_of(m));
        launch_reset_requests(c);
        launch_new_games(c, t.gids + (size_t)m * gcap, gcap, t.gstr + (size_t)m * gcap, nullptr, nullptr);
        RUN_EVAL(c, evaluator, gcap);
        launch_apply(c, t.gids + (size_t)m * gcap, gcap, kApplyNewGame);
    }
    launch_tourney_gather(c, t, 0);
    const int rounds = (count + batch_size - 1) / batch_size;  // parallel_mcts_executor.rs:39-42,207
    std::vector<int32_t> back((size_t)n + 1, (n - 1) * Q);     // {device error word, each participant's group size}
    back[0] = 0;
    const uint64_t naive_key = mix64(seed ^ kNaiveKey);
    const int32_t *size = back.data() + 1;
    std::vector<int> movers;
    int64_t n_moves = 0, syncs = 0;
    // a game ends after at most 81 moves; a device error (out of node slots, a non-finite network output, a refused move)
    // ends the tournament at the half-move that raised it
    for (int half = 0; back[0] == 0 && half < kCells; ++half) {
        movers.clear();
        for (int m = 0; m < n; ++m)
            if (size[m] > 0) movers.push_back(m);
        if (movers.empty()) break;
        // the naive player searches nothing: its half-move is one launch on lane 0 in the last stage, and the models' groups
        // alternate over the lanes as they would without it
        const int naive_moves = naive && size[0] > 0 ? 1 : 0;
        const int lanes = two_lanes && movers.size() - naive_moves >= 2 ? 2 : 1;
        if (lanes == 2) lanes_fork(c);
        for (int stage = 0; stage < rounds + 2 && rc == OMK_OK; ++stage)
            for (size_t k = 0; k < movers.size() && rc == OMK_OK; ++k) {
                const int m = movers[k];
                if (naive && m == 0) {
                    if (stage == rounds + 1) launch_tourney_naive_move(c, t, half, size[0], naive_key);
                    continue;
                }
                const size_t g0 = (size_t)m * gcap;
                LaneScope lane(c, lanes == 2 ? (int)((k - naive_moves) % 2) : 0, 0);
                ModelScope model(c, slot_of(m));
                rc = match_stage(c, stage, rounds, half, t.gids + g0, size[m], t.gact + g0, t.gst + g0, t.gost + g0, batch_size, epsilon,
                                 alpha, evaluator);
            }
        if (lanes == 2) lanes_join(c);  // on an error too: nothing queued on lane 1 is left unordered with the main stream
        if (rc) return rc;
        launch_tourney_advance(c, t, half);
        launch_tourney_gather(c, t, half + 1);
        for (int m : movers) n_moves += size[m];
        // the half-move's one host round trip: the group sizes size the next launches
        CK(copy_d2h(c, back.data(), t.back, sizeof(int32_t) * back.size(), c->stream));
        CK(cudaStreamSynchronize(c->stream));
        ++syncs;
    }
    fold_requests(c);
    CK(cudaMemcpyAsync(sims + 2, c->dev_sims, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev1, c->stream));
    std::vector<uint8_t> host(out_bytes);
    CK(copy_d2h(c, host.data(), base, out_bytes, c->stream));
    rc = check_device_error(c);  // (synchronises the stream)
    ++syncs;
    if (rc) return rc;
    const unsigned long long *h_sims = reinterpret_cast<const unsigned long long *>(host.data());
    memcpy(out_result, host.data() + off_cnt, 12 * (size_t)P);
    if (out_status) memcpy(out_status, host.data() + off_fin, G);
    if (out_moves) memcpy(out_moves, host.data() + off_moves, G * kCells);
    if (out_stats) {
        out_stats[0] = (int64_t)(h_sims[2] - h_sims[0]);
        out_stats[1] = (int64_t)(h_sims[3] - h_sims[1]);
        out_stats[2] = n_moves;
        out_stats[3] = syncs;
    }
    if (out_gpu_ms) CK(cudaEventElapsedTime(out_gpu_ms, c->ev0, c->ev1));
    return OMK_OK;
}

extern "C" int32_t omk_tournament(omk_ctx *c, int32_t n_models, const int32_t *slots, int32_t pairs, int32_t first_tree, int32_t count,
                                  int32_t batch_size, float epsilon, float alpha, int32_t evaluator, int32_t *out_result,
                                  int8_t *out_moves, int8_t *out_status, int64_t *out_stats, float *out_gpu_ms) {
    return tournament(c, false, n_models, slots, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, 0, out_result,
                      out_moves, out_status, out_stats, out_gpu_ms);
}

extern "C" int32_t omk_tournament_naive(omk_ctx *c, int32_t n_models, const int32_t *slots, int32_t pairs, int32_t first_tree,
                                        int32_t count, int32_t batch_size, float epsilon, float alpha, int32_t evaluator, uint64_t seed,
                                        int32_t *out_result, int8_t *out_moves, int8_t *out_status, int64_t *out_stats,
                                        float *out_gpu_ms) {
    return tournament(c, true, n_models, slots, pairs, first_tree, count, batch_size, epsilon, alpha, evaluator, seed, out_result,
                      out_moves, out_status, out_stats, out_gpu_ms);
}
