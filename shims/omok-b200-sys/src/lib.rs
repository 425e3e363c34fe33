//! Raw bindings of include/omok_b200.h (one declaration per entry point, same order as the header) and the process-wide
//! context the safe crates share.  NOT COMPILED in the build image of this repository (no Rust toolchain): see ../README.md.
#![allow(non_camel_case_types)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_void};
use std::sync::{Mutex, OnceLock};

pub const OMK_CELLS: usize = 81;
pub const OMK_NONE: i8 = -1;
pub const OMK_OK: i32 = 0;
pub const OMK_ERR_INVALID: i32 = -1;
pub const OMK_ERR_CUDA: i32 = -2;
pub const OMK_ERR_CAPACITY: i32 = -3;
pub const OMK_ERR_STATE: i32 = -4;
pub const OMK_ERR_NUMERIC: i32 = -5;
pub const OMK_EVAL_NET: i32 = 0;
pub const OMK_EVAL_HASH: i32 = 1;
pub const OMK_SAMPLE_BEST: u8 = 0;
pub const OMK_SAMPLE_BOLTZMANN: u8 = 1;
pub const OMK_TURN_MODE_PLAYER: i32 = 0;
pub const OMK_TURN_MODE_OPPONENT: i32 = 1;
pub const OMK_NET_TENSORS: usize = 31;
pub const OMK_K_COUNT: usize = 8;

#[repr(C)]
pub struct omk_ctx {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct omk_selfplay_config {
    pub n_games: i32,
    pub count: i32,
    pub batch_size: i32,
    pub epsilon: f32,
    pub alpha: f32,
    pub temperature: f32,
    pub temperature_threshold: i32,
    pub evaluator: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct omk_selfplay_stats {
    pub simulations: i64,
    pub positions: i64,
    pub nn_evals: i64,
    pub games_finished: i64,
    pub h2d_bytes: i64,
    pub d2h_bytes: i64,
    pub gpu_ms: f32,
    pub kind_ms: [f32; OMK_K_COUNT],
    pub kind_launches: [i64; OMK_K_COUNT],
}

extern "C" {
    pub fn omk_last_error() -> *const c_char;
    pub fn omk_version() -> i32;
    // context
    pub fn omk_ctx_create(device: i32, capacity_envs: i32, capacity_trees: i32, capacity_nodes: i32, seed: u64, out: *mut *mut omk_ctx) -> i32;
    pub fn omk_ctx_destroy(ctx: *mut omk_ctx) -> i32;
    pub fn omk_ctx_synchronize(ctx: *mut omk_ctx) -> i32;
    pub fn omk_ctx_stream(ctx: *mut omk_ctx) -> *mut c_void;
    pub fn omk_ctx_launch_count(ctx: *mut omk_ctx) -> i64;
    pub fn omk_ctx_transfer_bytes(ctx: *mut omk_ctx, out_h2d: *mut i64, out_d2h: *mut i64) -> i32;
    // network (alpha-zero/src/agent_model.rs:105-134, network.rs:51-262)
    pub fn omk_net_load_params(ctx: *mut omk_ctx, tensors: *const *const f32, lens: *const i64) -> i32;
    pub fn omk_net_get_params(ctx: *mut omk_ctx, tensors: *const *mut f32, lens: *const i64) -> i32;
    pub fn omk_net_init_random(ctx: *mut omk_ctx, seed: u64) -> i32;
    pub fn omk_net_eval(ctx: *mut omk_ctx, boards: *const u8, turns: *const u8, n: i32, mode: i32, out_p: *mut f32, out_v: *mut f32) -> i32;
    // trainer step (alpha-zero/src/agent_model.rs:136-168)
    pub fn omk_train_step(ctx: *mut omk_ctx, images: *const f32, pi: *const f32, z: *const f32, n: i32, out_losses: *mut f32) -> i32;
    pub fn omk_train_backward(ctx: *mut omk_ctx, images: *const f32, pi: *const f32, z: *const f32, n: i32, out_grads_device: *mut *mut c_void, out_count: *mut i64) -> i32;
    pub fn omk_train_apply(ctx: *mut omk_ctx, out_losses: *mut f32) -> i32;
    pub fn omk_train_get_grads(ctx: *mut omk_ctx, tensors: *const *mut f32, lens: *const i64) -> i32;
    pub fn omk_train_reset_optimizer(ctx: *mut omk_ctx) -> i32;
    pub fn omk_train_get_optimizer(ctx: *mut omk_ctx, accum: *const *mut f32, accum_update: *const *mut f32, lens: *const i64) -> i32;
    pub fn omk_train_set_optimizer(ctx: *mut omk_ctx, accum: *const *const f32, accum_update: *const *const f32, lens: *const i64) -> i32;
    pub fn omk_train_comm_unique_id(ctx: *mut omk_ctx, out_id: *mut u8) -> i32;
    pub fn omk_train_comm_init(ctx: *mut omk_ctx, id: *const u8, nranks: i32, rank: i32) -> i32;
    pub fn omk_train_comm_destroy(ctx: *mut omk_ctx) -> i32;
    pub fn omk_net_eval_images(ctx: *mut omk_ctx, images: *const f32, n: i32, out_p: *mut f32, out_v: *mut f32) -> i32;
    // diagnostics
    pub fn omk_debug_set_fc0_mode(ctx: *mut omk_ctx, mode: i32) -> i32;
    pub fn omk_debug_set_tower_mode(ctx: *mut omk_ctx, mode: i32) -> i32;
    pub fn omk_debug_set_fc0_chunk(ctx: *mut omk_ctx, k_blocks: i32) -> i32;
    pub fn omk_debug_set_fc0_balance(ctx: *mut omk_ctx, on: i32) -> i32;
    pub fn omk_debug_tower_timing(ctx: *mut omk_ctx, out64: *mut i64) -> i32;
    pub fn omk_debug_get_buffer(ctx: *mut omk_ctx, which: i32, out: *mut f32, count: i64) -> i32;
    pub fn omk_debug_set_lane_min_trees(ctx: *mut omk_ctx, min_trees: i32) -> i32;
    // environment (environment/src/lib.rs:62-193)
    pub fn omk_env_reset(ctx: *mut omk_ctx, ids: *const i32, n: i32) -> i32;
    pub fn omk_env_step(ctx: *mut omk_ctx, ids: *const i32, actions: *const u8, n: i32, out_status: *mut i8, out_legal: *mut u32) -> i32;
    pub fn omk_env_step_device(ctx: *mut omk_ctx, actions_device: *const u8, n: i32, out_status_device: *mut i8, out_legal_device: *mut u32) -> i32;
    pub fn omk_env_get(ctx: *mut omk_ctx, ids: *const i32, n: i32, out_boards: *mut u8, out_turns: *mut u8, out_legal_counts: *mut u16) -> i32;
    pub fn omk_env_set(ctx: *mut omk_ctx, ids: *const i32, n: i32, boards: *const u8, turns: *const u8) -> i32;
    pub fn omk_env_encode(ctx: *mut omk_ctx, ids: *const i32, n: i32, mode: i32, out: *mut f32) -> i32;
    pub fn omk_env_random_playout(ctx: *mut omk_ctx, n: i32, plies: i32, out_actions: *mut u8, out_status: *mut i8) -> i32;
    // tree pool (alpha-zero/src/agent.rs, parallel_mcts_executor.rs, mcts_executor.rs; mcts/src/*.rs)
    pub fn omk_pool_new_games(ctx: *mut omk_ctx, ids: *const i32, n: i32, streams: *const u32, evaluator: i32) -> i32;
    pub fn omk_pool_search(ctx: *mut omk_ctx, ids: *const i32, n: i32, count: i32, batch_size: i32, epsilon: f32, alpha: f32, evaluator: i32) -> i32;
    pub fn omk_search_set_virtual_loss(ctx: *mut omk_ctx, enabled: i32) -> i32;
    pub fn omk_pool_sample(ctx: *mut omk_ctx, ids: *const i32, n: i32, modes: *const u8, temperatures: *const f32, out_actions: *mut i32, out_policy: *mut f32) -> i32;
    pub fn omk_pool_policy(ctx: *mut omk_ctx, ids: *const i32, n: i32, out_policy: *mut f32, out_valid: *mut u8) -> i32;
    pub fn omk_pool_ensure_action(ctx: *mut omk_ctx, ids: *const i32, actions: *const i32, n: i32, evaluator: i32) -> i32;
    pub fn omk_pool_play(ctx: *mut omk_ctx, ids: *const i32, actions: *const i32, n: i32, out_status: *mut i8) -> i32;
    pub fn omk_pool_get_env(ctx: *mut omk_ctx, id: i32, out_board: *mut u8, out_turn: *mut u8, out_legal_count: *mut u16) -> i32;
    pub fn omk_pool_get_envs(ctx: *mut omk_ctx, ids: *const i32, n: i32, out_boards: *mut u8, out_turns: *mut u8, out_legal_counts: *mut u16, out_status: *mut i8) -> i32;
    pub fn omk_pool_root_stats(ctx: *mut omk_ctx, id: i32, out_n: *mut u64, out_w: *mut f32, out_p: *mut f32, out_status: *mut i32, out_policy: *mut f32) -> i32;
    pub fn omk_pool_root_children(ctx: *mut omk_ctx, id: i32, out_actions: *mut i32, out_n: *mut u64, out_w: *mut f32, out_p: *mut f32, out_len: *mut i32) -> i32;
    pub fn omk_pool_tree_info(ctx: *mut omk_ctx, id: i32, out_nodes: *mut i32, out_rng_counter: *mut u32) -> i32;
    // device-resident self-play driver (src/trainer.rs:86-204)
    pub fn omk_selfplay_begin(ctx: *mut omk_ctx, cfg: *const omk_selfplay_config) -> i32;
    pub fn omk_selfplay_run(ctx: *mut omk_ctx, plies: i32, profile: i32, out_boards: *mut u8, out_policy: *mut f32, out_status: *mut i8, out_actions: *mut i32, stats: *mut omk_selfplay_stats) -> i32;
    pub fn omk_selfplay_set_model(ctx: *mut omk_ctx, slot: i32) -> i32;
    // device replay memory (src/trainer.rs:27,206-352) and the training phase on it
    pub fn omk_replay_reset(ctx: *mut omk_ctx, capacity: i64) -> i32;
    pub fn omk_replay_info(ctx: *mut omk_ctx, out_len: *mut i64, out_rows_added: *mut i64, out_episodes: *mut i64) -> i32;
    pub fn omk_replay_get(ctx: *mut omk_ctx, rows: *const i64, n: i32, out_boards: *mut u8, out_turns: *mut u8, out_policy: *mut f32, out_z: *mut f32) -> i32;
    pub fn omk_replay_append(ctx: *mut omk_ctx, boards: *const u8, turns: *const u8, policy: *const f32, z: *const f32, n: i32, episodes: i64) -> i32;
    pub fn omk_train_replay(ctx: *mut omk_ctx, seed: u64, first_step: i64, steps: i32, n: i32, out_losses: *mut f32, out_rows: *mut i64) -> i32;
    pub fn omk_replay_score(ctx: *mut omk_ctx, slot: i32, rows: *const i64, first: i64, n: i32, out_means: *mut c_void, out_row_p_loss: *mut f32, out_row_v_loss: *mut f32, out_row_top1: *mut u8) -> i32;
    // evaluation against the naive player (src/trainer.rs:487-603)
    pub fn omk_naive_move(ctx: *mut omk_ctx, boards: *const u8, turns: *const u8, n: i32, seed: u64, streams: *const u32, out_actions: *mut i32, out_forced: *mut u8) -> i32;
    pub fn omk_eval_naive(ctx: *mut omk_ctx, episodes: i32, first_tree: i32, count: i32, batch_size: i32, epsilon: f32, alpha: f32, evaluator: i32, seed: u64, out_result: *mut i32, out_moves: *mut i8, out_status: *mut i8, out_stats: *mut i64, out_gpu_ms: *mut f32) -> i32;
    // the opponent network and the arena (benchmark/src/main.rs:14-108)
    pub fn omk_opponent_load_params(ctx: *mut omk_ctx, tensors: *const *const f32, lens: *const i64) -> i32;
    pub fn omk_opponent_from_net(ctx: *mut omk_ctx) -> i32;
    pub fn omk_opponent_eval(ctx: *mut omk_ctx, boards: *const u8, turns: *const u8, n: i32, mode: i32, out_p: *mut f32, out_v: *mut f32) -> i32;
    pub fn omk_match(ctx: *mut omk_ctx, pairs: i32, first_tree: i32, count: i32, batch_size: i32, epsilon: f32, alpha: f32, evaluator: i32, out_result: *mut i32, out_moves: *mut i8, out_status: *mut i8, out_stats: *mut i64, out_gpu_ms: *mut f32) -> i32;
    // model slots and the tournament (a round-robin of the arena)
    pub fn omk_model_load_params(ctx: *mut omk_ctx, slot: i32, tensors: *const *const f32, lens: *const i64) -> i32;
    pub fn omk_model_from_net(ctx: *mut omk_ctx, slot: i32) -> i32;
    pub fn omk_model_get_params(ctx: *mut omk_ctx, slot: i32, tensors: *const *mut f32, lens: *const i64) -> i32;
    pub fn omk_model_eval(ctx: *mut omk_ctx, slot: i32, boards: *const u8, turns: *const u8, n: i32, mode: i32, out_p: *mut f32, out_v: *mut f32) -> i32;
    pub fn omk_tournament(ctx: *mut omk_ctx, n_models: i32, slots: *const i32, pairs: i32, first_tree: i32, count: i32, batch_size: i32, epsilon: f32, alpha: f32, evaluator: i32, out_result: *mut i32, out_moves: *mut i8, out_status: *mut i8, out_stats: *mut i64, out_gpu_ms: *mut f32) -> i32;
    pub fn omk_tournament_naive(ctx: *mut omk_ctx, n_models: i32, slots: *const i32, pairs: i32, first_tree: i32, count: i32, batch_size: i32, epsilon: f32, alpha: f32, evaluator: i32, seed: u64, out_result: *mut i32, out_moves: *mut i8, out_status: *mut i8, out_stats: *mut i64, out_gpu_ms: *mut f32) -> i32;
}

/// The message of the last failing call on this thread.
pub fn last_error() -> String {
    unsafe { CStr::from_ptr(omk_last_error()).to_string_lossy().into_owned() }
}

/// Process-wide context: one CUDA device, env / tree slots handed out from free lists.  A context is used by one host
/// thread at a time (include/omok_b200.h), hence the mutex around every call made through `with`.
pub struct Context {
    raw: *mut omk_ctx,
    free_envs: Vec<i32>,
    free_trees: Vec<i32>,
}
unsafe impl Send for Context {}

static CTX: OnceLock<Mutex<Context>> = OnceLock::new();

fn env_or<T: std::str::FromStr>(name: &str, default: T) -> T {
    std::env::var(name).ok().and_then(|v| v.parse().ok()).unwrap_or(default)
}

impl Context {
    fn create() -> Context {
        let (device, envs, trees, nodes, seed) = (
            env_or("OMOK_B200_DEVICE", 0i32),
            env_or("OMOK_B200_ENVS", 65536i32),
            env_or("OMOK_B200_TREES", 4096i32),
            env_or("OMOK_B200_NODES", 4096i32),
            env_or("OMOK_B200_SEED", 0u64),
        );
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { omk_ctx_create(device, envs, trees, nodes, seed, &mut raw) };
        assert!(rc == OMK_OK, "omk_ctx_create: {}", last_error());
        Context { raw, free_envs: (0..envs).rev().collect(), free_trees: (0..trees).rev().collect() }
    }
    pub fn raw(&self) -> *mut omk_ctx {
        self.raw
    }
    pub fn take_env(&mut self) -> i32 {
        self.free_envs.pop().expect("env pool exhausted: raise OMOK_B200_ENVS")
    }
    pub fn give_env(&mut self, slot: i32) {
        self.free_envs.push(slot)
    }
    pub fn take_tree(&mut self) -> i32 {
        self.free_trees.pop().expect("tree pool exhausted: raise OMOK_B200_TREES")
    }
    pub fn give_tree(&mut self, slot: i32) {
        self.free_trees.push(slot)
    }
}

/// Runs `f` with the locked process-wide context.
pub fn with<R>(f: impl FnOnce(&mut Context) -> R) -> R {
    let m = CTX.get_or_init(|| Mutex::new(Context::create()));
    let mut guard = m.lock().unwrap();
    f(&mut guard)
}

/// `Ok(())` for OMK_OK, the library's message otherwise.
pub fn check(rc: i32) -> Result<(), String> {
    if rc == OMK_OK {
        Ok(())
    } else {
        Err(format!("libomok_b200 error {rc}: {}", last_error()))
    }
}
