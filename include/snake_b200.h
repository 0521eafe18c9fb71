/*
 * snake_b200.h — C ABI of libsnake_b200.so, the B200-native batched Snake environment
 * and Laplace D-matrix kernels.
 *
 * This is the drop-in boundary for the environment hot path of
 * lucagiorgetti/Laplace-DQN-Snake-game (Julia).  The reference has no FFI of its own; each
 * entry point below names the Julia function (file:line in the reference repository) it
 * replaces.  A Julia host binds these with `ccall` (see INTEGRATION.md and
 * laplace-dqn-snake-game_b200/julia/SnakeB200.jl); the tests and bench bind the identical
 * symbols with ctypes.
 *
 * Conventions
 *   - every function returns int: 0 = SNK_OK, < 0 = error (snk_last_error() has the text);
 *     no C++ exception crosses this boundary;
 *   - pointers are DEVICE pointers unless the function name ends in `_host`;
 *   - N = number of envs of the handle; per-env arrays are length N, `(3,N)` arrays are
 *     3*N elements with the 3 contiguous (Julia column-major), observations are
 *     `(10,10,2,N)` column-major exactly as `stack_exp` builds them (utils.jl:348-362):
 *     element (r,c,f,n), 1-based, lives at (r-1) + 10(c-1) + 100(f-1) + 200(n-1);
 *     frame f=1 is the older board, f=2 the newer one;
 *   - calls enqueue work on the handle's CUDA stream and return; snk_sync() waits.  This includes
 *     snk_step_fused_host / snk_step_fused_store_host: their host buffers are read and written
 *     asynchronously — call snk_sync() before reading an output or reusing an input buffer.
 *     The per-call getters whose names end in `_host` (snk_state_host, snk_losing_mask_host, ...)
 *     return when the data has arrived;
 *   - every call runs on its handle's device and restores the caller's current device; the stateless
 *     entry points (snk_masked_target, snk_center_columns, snk_gram*, ...) run on the device that
 *     owns their workspace / output pointer;
 *   - one handle per host thread; there is no hidden global state besides the
 *     thread-local error string and the tile-engine switch snk_gram_config;
 *   - there is no CPU fallback: without a CUDA device snk_create fails.
 *
 * Codes
 *   direction: 0=U(-1,0) 1=D(+1,0) 2=L(0,-1) 3=R(0,+1)             (utils.jl:8)
 *   action index 0..2: position in available_actions(game)          (utils.jl:7-10)
 *   board cell: -1 wall, 0 empty, 1 snake, 2 food                   (structs.jl:34-51)
 *   rewards: +1f0 eat, -1f0 loss, -0.01f0 otherwise                 (structs.jl:89-91)
 */
#ifndef SNAKE_B200_H
#define SNAKE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNK_VERSION 200

#if defined(__GNUC__)
#define SNK_API __attribute__((visibility("default")))
#else
#define SNK_API
#endif

/* return codes */
#define SNK_OK 0
#define SNK_ERR_INVALID (-1)   /* bad argument */
#define SNK_ERR_CUDA (-2)      /* a CUDA runtime call failed */
#define SNK_ERR_NODEVICE (-3)  /* no CUDA device / not a Blackwell part */
#define SNK_ERR_UNSUPPORTED (-4)
#define SNK_ERR_TIMEOUT (-5)   /* a peer of the row-sharded Gram, a learner group or a replay group did not arrive in time */

/* snk_create flags */
#define SNK_AUTO_RESET 1u      /* a lost env is re-initialised (a fresh SnakeGame(), utils.jl:199) after its terminal outputs */

/* per-env sticky error bits (snk_get_error_flags) */
#define SNK_ENV_ERR_FOOD 1u    /* sample_food! had empty cells but no usable list entry: BoundsError in the reference (utils.jl:23,37) */
#define SNK_ENV_ERR_ACTION 2u  /* action index > 2 or direction > 3 was passed; treated as 0 */

/* observation formats */
#define SNK_OBS_NONE 0
#define SNK_OBS_F32 1          /* Float32.(state), utils.jl:361-362: 800 B/env */
#define SNK_OBS_I8 2           /* same values as int8: 200 B/env */
#define SNK_OBS_I64 3          /* game.state::Array{Int,4}, structs.jl:17: 1600 B/env */
#define SNK_OBS_PACKED2 4      /* 2 bits/cell, 4 cells/byte (cell j of a byte in bits 2j..2j+1), codes 0,1,2 and 3 = wall: 50 B/env */
/* SNK_OBS_BITS: 24 B/env, lossless — the two boards as bit-boards plus the step's scalars (little endian):
 *   [0,8)   u64 snake bitmap of the OLDER board: bit (r-1) + 8 (c-1) <=> interior cell (r, c), 0-based, 1 <= r, c <= 8
 *   [8,16)  u64 snake bitmap of the NEWER board (without the head cell below when that lies on a wall)
 *   [16] food of the older board, [17] food of the newer board, [18] head of the newer board: cell (r, c) as r | c << 4,
 *        0-based full-board coordinates; food byte 0 = no food on the board
 *   [19] bits 0-2 next_is_suicidal of the three offered moves, bit 3 done, bits 4-5 the action taken (index or direction)
 *   [20,24) Float32 reward
 * board(r, c) = -1 on the wall ring, 1 where the bitmap (or, newer board, the head: update_board! overwrites the wall cell on
 * a wall death, utils.jl:48-50) is set, 2 on the food cell unless the snake is there, else 0.  Accepted by snk_step*,
 * snk_step_fused*, snk_state*, snk_patch_reset_obs (not by snk_rollout); the host mirrors decode it (unpack_bits). */
#define SNK_OBS_BITS 5

typedef struct snk_env *snk_handle;

/* ---- lifecycle: SnakeGame(board_size=10, n_frames=2)  structs.jl:33-99 ------------------- */
SNK_API int snk_create(snk_handle *out, int64_t n_envs, int device, uint32_t flags);
SNK_API int snk_destroy(snk_handle h);
/* every env back to the constructor state (R1): walls, food (4,5), snake [(8,2),(9,2)], prev_dir U */
SNK_API int snk_reset(snk_handle h);
/* food_list injection (structs.jl:70).  cells_rc_host: n pairs (row, col), 1-based, 2..9; n <= 64.
 * Default = the 50 cells Xoshiro(42) yields (snk_default_food_list_host).  The table is swapped immediately, but the
 * consumed-entry bitmaps of running episodes refer to the old list: call snk_reset right after. */
SNK_API int snk_set_food_list_host(snk_handle h, const uint8_t *cells_rc_host, int n);
SNK_API int snk_default_food_list_host(uint8_t *cells_rc_host /* 100 bytes */, int *n);
/* A handle starts on its own non-blocking stream.  snk_set_stream adopts an external one (cudaStream_t /
 * CUstream, e.g. torch's current stream; NULL = the legacy default stream); snk_use_own_stream goes back. */
SNK_API int snk_set_stream(snk_handle h, void *cuda_stream);
SNK_API int snk_use_own_stream(snk_handle h);
SNK_API int snk_get_stream(snk_handle h, void **cuda_stream);
/* seed of the internal counter-based generator used when draws are not injected */
SNK_API int snk_set_seed(snk_handle h, uint64_t seed);
SNK_API int snk_sync(snk_handle h);
SNK_API int64_t snk_num_envs(snk_handle h);
SNK_API const char *snk_last_error(void);
SNK_API int snk_version(void);

/* ---- available_actions(game)  utils.jl:7-10 ---------------------------------------------- */
SNK_API int snk_available_actions(snk_handle h, uint8_t *dirs_3xN);
SNK_API int snk_available_actions_host(snk_handle h, uint8_t *dirs_3xN_host);

/* ---- step!(game, action)  utils.jl:100-109 (+ grow_maybe!, sample_food!, check_collision,
 *      update_board!, move_wrapper!: utils.jl:13-96) ---------------------------------------
 * act_idx: 0..2 into available_actions (what the Q-net's argmax means, utils.jl:165-167).
 * reward: game.reward (exact Float32 bit patterns), done: game.lost.  Either may be NULL.
 * A lost env without SNK_AUTO_RESET is left untouched and reports reward 0, done 1. */
SNK_API int snk_step(snk_handle h, const uint8_t *act_idx, float *reward, uint8_t *done);
/* absolute directions as play_snake.jl:96-111 sends them; a reverse move loses (utils.jl:57) */
SNK_API int snk_step_abs(snk_handle h, const uint8_t *dir, float *reward, uint8_t *done);

/* ---- the fused hot path: one kernel per rollout step -------------------------------------
 * = epsilon_greedy (optional) + step! + virtual_step + assemble_states_vector's next_state +
 *   Float32.() of stack_exp, for all N envs  (utils.jl:153-172, 100-109, 112-132, 141-149, 361-362).
 * Inputs:  q != NULL  -> actions are chosen here by epsilon_greedy from q (3,N) f32 with
 *                        eps; u (N) f32 and ridx (N) u8 in 0..2 are the injected draws
 *                        `Float32(rand())` and the index `rand(av_actions)` picks; if u / ridx
 *                        are NULL they come from the internal generator.  act_idx then is an
 *                        optional OUTPUT (N) u8.
 *          q == NULL  -> act_idx (N) u8 is the INPUT action index.
 *          The internal generator is keyed by (seed, env, number of step calls so far); the call count is a launch
 *          argument, so a CUDA graph replays the SAME draws: inject u / ridx when capturing steps into a graph.
 * Outputs (any may be NULL): reward (N) f32, done (N) u8,
 *          obs: next_state (board_{t-1}, board_t) in obs_fmt, the terminal pair when done;
 *          mask (3,N) u8: next_is_suicidal (trues(3) when done);
 *          ep_return (N) f32: running Float32 episode reward (utils.jl:200,207) incl. this step;
 *          ep_score (N) i32: game.score after this step. */
SNK_API int snk_step_fused(snk_handle h, const float *q, float eps, const float *u, const uint8_t *ridx,
                   uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt,
                   uint8_t *mask, float *ep_return, int32_t *ep_score);
/* same call with HOST buffers (pinned memory recommended: snk_host_alloc): env chunks are pipelined three deep — the
 * inputs of chunk c+1 go up while the kernel of chunk c runs and the outputs of chunk c-1 come down.  ASYNCHRONOUS:
 * returns after enqueueing; snk_sync(h) before reading an output or overwriting an input.  The output copies run on a
 * copy stream of the handle: work enqueued afterwards on the handle's stream (a snk_replay_gather_host of the minibatch,
 * the Q-net forward of the next step) overlaps them; only snk_sync waits for them.  obs_fmt SNK_OBS_PACKED2
 * (50 B/env, lossless) is the format meant for this entry: the reference casts to Float32 only the 64 transitions a
 * minibatch samples (utils.jl:361-362) — snk_replay_gather_host does that for the device replay ring. */
SNK_API int snk_step_fused_host(snk_handle h, const float *q, float eps, const float *u, const uint8_t *ridx,
                        uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt,
                        uint8_t *mask, float *ep_return, int32_t *ep_score);
/* T steps of step! + virtual_step + next_state in ONE launch, for action streams known up front
 * (play_episode's actions_list mode, utils.jl:209-219; BASELINE config 2 "uniform random actions").  Small batches
 * are launch-latency bound; here every env stays in registers across the T steps.  Step-major arrays:
 * act (T,N) u8 indices (or absolute directions if is_abs), reward (T,N) f32, done (T,N) u8, mask (T,3,N) u8,
 * obs (T, 10,10,2,N) in obs_fmt, ep_return / ep_score (T,N).  Outputs may be NULL. */
SNK_API int snk_rollout_fused(snk_handle h, const uint8_t *act_TxN, int64_t T, int is_abs, float *reward, uint8_t *done,
                              void *obs, int obs_fmt, uint8_t *mask, float *ep_return, int32_t *ep_score);
/* profiling aid: device buffer of 8 int64 that receives cycle counts of CTA 0 of the small-batch rollout kernel on every later
 * snk_rollout_fused ([0] logic warp total, [1] its wait for the expander warps, [2] expander wait for the logic warp,
 * [3] losing mask + boards, [4] observation expansion); NULL switches it off */
SNK_API int snk_debug_rollout_timing(long long *device_buf);
SNK_API int snk_host_alloc(void **p, size_t bytes);   /* pinned host memory */
SNK_API int snk_host_free(void *p);
/* device memory for the outputs of the fused step.  With SNK_ALLOC_COMPRESSIBLE, on a device that supports it
 * (snk_compression_supported), the memory is created with generic L2 compression (cuMemCreate, CU_MEM_ALLOCATION_COMP_GENERIC,
 * size rounded up to the allocation granularity, 2 MB on B200): lossless, every kernel and copy sees the same bytes, but lines
 * of few distinct words - the Float32 observations - cross the DRAM bus compressed, so k_step writing into it is faster.
 * Otherwise, or when the driver hands out memory that is not compressible, it is cudaMalloc memory.  *compressible (may be
 * NULL) reports which one it is.  snk_device_free synchronises the device before it unmaps compressible memory: not for use
 * inside a CUDA graph capture. */
#define SNK_ALLOC_COMPRESSIBLE 1u
SNK_API int snk_device_alloc(void **p, size_t bytes, int device, uint32_t flags, int *compressible);
SNK_API int snk_device_free(void *p);
SNK_API int snk_compression_supported(int device, int *yes);

/* ---- assemble_state! / assemble_states_vector  utils.jl:135-149 --------------------------- */
/* current two-frame state (board_{t-1}, board_t) of every env, in obs_fmt */
SNK_API int snk_state(snk_handle h, void *obs, int obs_fmt);
SNK_API int snk_state_host(snk_handle h, void *obs_host, int obs_fmt);        /* returns when the data has arrived */
/* obs = the next_state output of the fused step that produced `done`: rows of envs that step re-initialised (done != 0,
 * SNK_AUTO_RESET) are overwritten with the constructor state (init, init) (structs.jl:53-55) — obs then is the acting
 * state of the next step for every env, without re-expanding all N (a batched play_episode loop, utils.jl:203-208) */
SNK_API int snk_patch_reset_obs(snk_handle h, const uint8_t *done, void *obs, int obs_fmt);

/* ---- virtual_step(game, model)  utils.jl:112-132 ------------------------------------------ */
/* next_is_suicidal for the CURRENT state: for each available action, would step! lose?
 * trues(3) for a lost env.  Includes the history-length rule (all true after 499 steps). */
SNK_API int snk_losing_mask(snk_handle h, uint8_t *mask_3xN);
SNK_API int snk_losing_mask_host(snk_handle h, uint8_t *mask_3xN_host);

/* ---- epsilon_greedy(game, model, eps)  utils.jl:153-172 ----------------------------------- */
/* out[i] = ridx[i] if u[i] < eps else argmax(q[:,i]) (Julia argmax: first maximum, NaN wins). */
SNK_API int snk_select_action(snk_handle h, const float *q_3xN, float eps, const float *u, const uint8_t *ridx,
                      uint8_t *act_idx_out);

/* ---- masked max-Q target  utils.jl:448-451 ------------------------------------------------ */
/* q_next[mask] .= fill; y = r + gamma * max_a q_next * (1 - done), evaluated in Float64 as the
 * reference's broadcast does (0.97 is a Float64 literal).  y_f64 and/or y_f32 (= Float32(y)) may be
 * NULL.  Stateless; runs on `cuda_stream` (NULL = default stream) of the current device. */
SNK_API int snk_masked_target(const float *q_next_3xB, const uint8_t *mask_3xB, const float *r, const uint8_t *done,
                      double gamma, float fill, double *y_f64, float *y_f32, int64_t B, void *cuda_stream);

/* ---- per-env scalars ---------------------------------------------------------------------- */
SNK_API int snk_get_score(snk_handle h, int32_t *score);          /* game.score  structs.jl:21 */
SNK_API int snk_get_done(snk_handle h, uint8_t *done);            /* game.lost   structs.jl:28 */
SNK_API int snk_get_error_flags(snk_handle h, uint8_t *flags);    /* SNK_ENV_ERR_* */
SNK_API int snk_get_steps(snk_handle h, int32_t *steps);          /* steps taken in the current episode */
/* the same into HOST arrays (game.score / game.lost as a Julia host reads them); return when the data has arrived */
SNK_API int snk_get_score_host(snk_handle h, int32_t *score_host);
SNK_API int snk_get_done_host(snk_handle h, uint8_t *done_host);
SNK_API int snk_get_error_flags_host(snk_handle h, uint8_t *flags_host);
SNK_API int snk_get_steps_host(snk_handle h, int32_t *steps_host);
/* number of envs with any error bit set (synchronises) */
SNK_API int snk_count_errors_host(snk_handle h, int64_t *count);

/* ---- checkpoints of a handle: save_trainer / load_trainer (utils.jl:408-418) -------------------------------------------
 * A blob (host memory, opaque, little endian) holds everything a later call on the handle depends on: a header (magic, format
 * version, N, the snk_create flags, seed, the call counter of the internal generator, the food list) and the raw state arrays
 * of the N envs — a handle loaded from it continues bit for bit like the one it was saved from.  snk_env_checkpoint_bytes gives
 * the size (176 + 52 N bytes); snk_env_save_host waits for the work enqueued on the handle's stream, copies and returns.
 * snk_env_load_host checks the header, then the blob's every env on the device (DESIGN §5e: coordinates, length, step count,
 * the direction chain against occupancy and tail, consumed food entries within the blob's list); only a blob that passes
 * replaces the handle's state, seed, counter and food list.  A refused blob (SNK_ERR_INVALID: wrong magic or version, a size
 * that is not the blob's, another N or auto-reset flag, an env that fails a rule — *first_bad_env (may be NULL) = the lowest
 * such env, else -1) leaves the handle as it was.  A blob saved on one device loads on another.  Both synchronise. */
SNK_API int snk_env_checkpoint_bytes(snk_handle h, size_t *bytes);
SNK_API int snk_env_save_host(snk_handle h, void *blob_host, size_t bytes);
SNK_API int snk_env_load_host(snk_handle h, const void *blob_host, size_t bytes, int64_t *first_bad_env);

/* ---- replay buffer  ReplayBuffer (structs.jl:104-116), store! / sample / stack_exp (utils.jl:265-383) -------
 * The ring lives on the device as one 128-byte record per transition (three 2-bit-plane boards + scalars);
 * snk_step_fused_store is snk_step_fused that additionally store!s every env's Experience in env order — the
 * same slots N sequential store! calls would use (push until full, then overwrite from position 1).
 * snk_replay_gather is stack_exp for the records at idx[0..B) (0-based slots): states / next_states
 * (10,10,2,B) Float32, actions (B) u8 0-based index into available_actions (utils.jl:363 stores it 1-based),
 * rewards (B) f32, dones (B) u8, suicidal_mask (3,B) u8.  Any output may be NULL.
 * snk_replay_sample_indices draws B distinct slots of the filled part (sample(rpb), utils.jl:280-287; the
 * reference's StatsBase draw stream is not reproduced — pass your own idx to snk_replay_gather for parity). */
typedef struct snk_replay_s *snk_replay;
SNK_API int snk_replay_create(snk_replay *out, int64_t capacity, int device);
SNK_API int snk_replay_destroy(snk_replay r);
SNK_API int snk_replay_clear(snk_replay r);                                     /* empty_buffer!  utils.jl:311-314 */
SNK_API int snk_replay_length(snk_replay r, int64_t *length, int64_t *position);  /* length(rpb), rpb.position (1-based) */
SNK_API int snk_step_fused_store(snk_handle h, snk_replay r, const float *q, float eps, const float *u, const uint8_t *ridx,
                                 uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask,
                                 float *ep_return, int32_t *ep_score);
SNK_API int snk_replay_gather(snk_replay r, const int64_t *idx, int64_t B, float *states, float *next_states,
                              uint8_t *actions, float *rewards, uint8_t *dones, uint8_t *mask, float *ep_return,
                              int32_t *score, void *cuda_stream);
/* host-buffer forms: the fused step + store! with HOST buffers (asynchronous like snk_step_fused_host), and stack_exp of
 * the slots idx_host[0..B) into HOST arrays (expanded to Float32 on the device, 1,613 B per sample over PCIe; returns
 * when the data has arrived) — together the data path of one train! iteration (utils.jl:436-443) for a host trainer */
SNK_API int snk_step_fused_store_host(snk_handle h, snk_replay r, const float *q, float eps, const float *u,
                                      const uint8_t *ridx, uint8_t *act_idx, float *reward, uint8_t *done, void *obs,
                                      int obs_fmt, uint8_t *mask, float *ep_return, int32_t *ep_score);
SNK_API int snk_replay_gather_host(snk_replay r, const int64_t *idx_host, int64_t B, float *states, float *next_states,
                                   uint8_t *actions, float *rewards, uint8_t *dones, uint8_t *mask, void *cuda_stream);
SNK_API int snk_replay_sample_indices(snk_replay r, uint64_t seed, int64_t B, int64_t *idx_out, void *cuda_stream);
SNK_API int snk_replay_bad_index_host(snk_replay r, int *flag);
/* checkpoints of the ring: save_buffer / load_buffer (utils.jl:316-340).  The blob: a header (magic, format version, capacity,
 * transitions stored, sample calls so far) and the min(stored, capacity) filled records (40 + 128 per record bytes).  Save and
 * load synchronise the ring's device first (the ring has no stream of its own).  Load checks every record's scalars on the
 * device (action index <= 2, done <= 1, mask bits <= 7, previous direction <= 3) and refuses as snk_env_load_host does:
 * *first_bad_slot = the lowest failing record (else -1), the ring left as it was. */
SNK_API int snk_replay_checkpoint_bytes(snk_replay r, size_t *bytes);
SNK_API int snk_replay_save_host(snk_replay r, void *blob_host, size_t bytes);
SNK_API int snk_replay_load_host(snk_replay r, const void *blob_host, size_t bytes, int64_t *first_bad_slot);
/* ---- the replay group: one minibatch drawn uniformly from the union of the rings of a box (DESIGN §5g) ----------------
 * A group has `world` ranks (1 .. 16), one snk_replay_group per rank, each wrapping that rank's ring.  batch_all[world]: every
 * rank's share B_q >= 1 of the minibatch, fixed at create and the same on every rank, as is `seed`.
 *   The union: the ranks' filled slots concatenated in rank order; union index u is slot u - (n_0 + ... + n_{q-1}) of rank q,
 *   with n_q = min(stored, capacity) of ring q when its stream reaches the call.  n = n_0 + ... + n_{R-1}.
 *   Call e (the group's draw counter, 0 at create) draws with key splitmix64(seed ^ splitmix64(e)), the key
 *   snk_replay_sample_indices derives from a ring's draw counter, and rank r takes the counters [off_r, off_r + B_r) of that
 *   permutation of [0, n), off_r = B_0 + ... + B_{r-1}.
 * So the ranks' outputs concatenated in rank order equal, bit for bit, snk_replay_sample_indices(seed, B_0 + ... + B_{R-1})
 * and snk_replay_gather on ONE full ring of capacity n that holds the ranks' filled records concatenated and whose draw counter
 * is e; world = 1 is snk_replay_sample_indices + snk_replay_gather on the ring itself.
 * snk_replay_group_sample writes this rank's B_r transitions in snk_replay_gather's layout, and idx_out (B_r int64) its global
 * union indices; every output may be NULL.  Ranks order themselves on the device, on cuda_stream (no host synchronisation):
 * the call waits until every ring is complete for call e, reads the records over peer memory, then waits until every rank has
 * read, so the rank's next store into its ring cannot overwrite a slot a peer still reads.  Every rank must call sample the same
 * number of times, and store into its ring only on the stream it samples on.  A call with B_0 + ... + B_{R-1} > n writes no
 * output and sets the flag status_host reports as SNK_ERR_INVALID; a wait that gives up after ~20 s sets SNK_ERR_TIMEOUT
 * (both flags stay set).  draws / set_draws: the draw counter, the only state of the group a checkpoint needs.
 * Set-up as for snk_qnet_group: create -> export_host (128 bytes: the ring's IPC handle and the flag block's) -> [every rank's
 * 128 bytes to every rank] -> connect_host(world x 128 bytes in rank order, own entry ignored); connect_local wires the groups
 * of ONE process (virtual ranks on one GPU, each on its own stream).  The ring must outlive its group. */
#define SNK_REPLAY_GROUP_HANDLE_BYTES 128
typedef struct snk_replay_group_s *snk_replay_group;
SNK_API int snk_replay_group_create(snk_replay_group *out, snk_replay r, int world, int rank, const int64_t *batch_all,
                                    uint64_t seed);
SNK_API int snk_replay_group_destroy(snk_replay_group g);
SNK_API int snk_replay_group_export_host(snk_replay_group g, uint8_t *handle128);
SNK_API int snk_replay_group_connect_host(snk_replay_group g, const uint8_t *handles_world_x_128, int n_handles);
SNK_API int snk_replay_group_connect_local(snk_replay_group g, const snk_replay_group *peers, int n_peers);
SNK_API int snk_replay_group_sample(snk_replay_group g, int64_t *idx_out, float *states, float *next_states, uint8_t *actions,
                                    float *rewards, uint8_t *dones, uint8_t *mask, float *ep_return, int32_t *score,
                                    void *cuda_stream);
SNK_API int snk_replay_group_draws(snk_replay_group g, uint64_t *draws);
SNK_API int snk_replay_group_set_draws(snk_replay_group g, uint64_t draws);
/* *timed_out: a wait gave up on a peer (SNK_ERR_TIMEOUT); *too_few: a call found B_0 + ... + B_{R-1} > n (SNK_ERR_INVALID).
 * Synchronises. */
SNK_API int snk_replay_group_status_host(snk_replay_group g, int *timed_out, int *too_few);

/* ---- Q-network forward  structs.jl:127-139; call sites utils.jl:165 (acting), 448 (t_net targets) -------------
 * Conv(3x3,2=>16,relu,pad 1) -> Conv(3x3,16=>32,relu,pad 1) -> Conv(6x6,32=>64,relu) -> flatten -> Dense(1600,64,relu)
 * -> Dense(64,3), Flux semantics (true convolution, WHCN, column-major flatten).  theta_host = Flux.destructure(q_net)
 * (181,395 Float32: per layer weight then bias, column-major) as compute_D.jl:43,68 takes it.  obs: (10,10,2,N) f32 as
 * snk_state / snk_step_fused emit it; q_out: (3,N) f32.  tcgen05 implicit-GEMM convolutions with FP32 accumulation;
 * `precision` chooses the operand format:
 *   SNK_QNET_F32   Float32-faithful (the reference network is Float32): weights and activations as fp16 (hi, lo) pairs
 *                  = 22 significant bits, all four partial products on the tensor cores.  Stated tolerance against a
 *                  Float64 evaluation: 2e-5 of max|Q|; argmax identical to it wherever the top-2 gap exceeds 1e-4 of
 *                  max|Q|.  Activations must stay inside the fp16 range (|x| <= 65504): snk_qnet_overflow_host tells.
 *   SNK_QNET_BF16  bf16 operands: 3-4x faster, 1.5e-2 of max|Q| — a greedy action can differ from the reference's; for
 *                  throughput studies, not for parity. */
#define SNK_QNET_BF16 0
#define SNK_QNET_F32 1
typedef struct snk_qnet_s *snk_qnet;
SNK_API int snk_qnet_create(snk_qnet *out, const float *theta_host, int64_t n_params, int device, int precision);
SNK_API int snk_qnet_destroy(snk_qnet q);
SNK_API int snk_qnet_forward(snk_qnet q, const float *obs_f32, int64_t N, float *q_out_3xN, void *cuda_stream);
SNK_API int snk_qnet_precision(snk_qnet q, int *precision);
/* SNK_QNET_F32: *flag = 1 if a forward since the last call produced an activation outside the fp16 range (its Q-values are
 * then not valid); reads and clears the flag, synchronises the device */
SNK_API int snk_qnet_overflow_host(snk_qnet q, int *flag);
/* ---- per-sample gradients of the DQN loss  utils.jl:452-466 (Flux.huber_loss(q_net(s)[a], y), delta = 1) ------------
 * Row i of J = d huber(q_net(s_i)[a_i], y_i) / d theta, theta in Flux.destructure order (181,395 columns) — the per-sample
 * term of the batch loss, without its 1/B.  BASELINE config 5b takes the Gram of these rows over the replay buffer.
 * states (10,10,2,B) f32 and actions (B) u8 0-based as snk_replay_gather returns them, targets (B) Float64 as
 * snk_masked_target returns them.  Outputs (each optional): the bf16 planes hi / lo = bf16(v - hi) with a row pitch of
 * pitch_elems (exactly what snk_gram_block / snk_gram_shard_run(A_rows = NULL) consume: snk_gram_shard_planes,
 * snk_gram_planes_layout), J_f32 (B x ldJ) Float32, loss (B) Float32.  Computed in FP32 from the Float32 weights whatever
 * the handle's forward precision is. */
SNK_API int snk_qnet_sample_grads(snk_qnet q, const float *states, const uint8_t *actions, const double *targets, int64_t B,
                                  void *hi, void *lo, int64_t pitch_elems, float *J_f32, int64_t ldJ, float *loss,
                                  void *cuda_stream);
/* ---- the learner  utils.jl:452-472 ------------------------------------------------------------------------------------
 * snk_qnet_train_step: Flux.gradient of mean(huber(q_net(s)[a], y)) + Flux.Optimise.update!(RMSProp(eta, rho, epsilon), θ, g)
 * on the device (utils.jl:452-466).  g = Float32(Σ_i J_i / B) with J_i the rows of snk_qnet_sample_grads, summed in Float64
 * in sample order; then acc = Float32(rho acc + (1 - rho) g g), θ -= Float32(g eta / (sqrt(acc) + epsilon)) in Float64 with
 * a Float32 sqrt (Flux.Optimise's promotions).  Inputs as for snk_qnet_sample_grads, B >= 1.  acc = the optimiser's state for
 * θ (181,395 f32, caller-owned, zero-initialised = a fresh RMSProp).  Every device layout of the handle (both forward
 * precisions, the gradient kernel's copy) follows the new θ.  grad_out (181,395 f32, g) and loss_out (1 f32, the batch mean of
 * the per-sample losses) are optional.  SNK_QNET_F32: a θ outside the fp16 range sets the snk_qnet_overflow_host flag.
 * snk_qnet_set_params: θ = theta_dev (181,395 f32 on the handle's device, e.g. another handle's snk_qnet_params), every
 * layout re-derived: update_target_net! (utils.jl:469-472).  snk_qnet_params: the handle's own θ, Flux.destructure order,
 * read-only; it changes with every train step.
 * Both updates enqueue on cuda_stream and return.  The caller orders a train step or set_params and any other call on the
 * same handle (forward, sample_grads, a set_params reading its θ): the same stream, or an event.  The next snk_qnet_forward
 * waits on the host for the update's copy of conv1's 304 weights (they are kernel parameters), so it fails with
 * SNK_ERR_INVALID inside a stream capture: run one forward after an update outside the capture. */
SNK_API int snk_qnet_train_step(snk_qnet q, const float *states, const uint8_t *actions, const double *targets, int64_t B,
                                float *acc, double eta, double rho, double epsilon, float *grad_out, float *loss_out,
                                void *cuda_stream);
SNK_API int snk_qnet_set_params(snk_qnet q, const float *theta_dev, void *cuda_stream);   /* update_target_net!, utils.jl:469-472 */
SNK_API int snk_qnet_params(snk_qnet q, const float **theta_dev);
/* ---- the data-parallel learner: one Q-net trained on every GPU of a box (DESIGN §5f) ----------------------------------
 * A group has `world` ranks (1 .. 16), one snk_qnet_group per rank, each wrapping a Q-net handle; all ranks' handles hold the
 * same θ.  snk_qnet_group_train_step(g, states, actions, targets, B_local, ...) takes the arguments of snk_qnet_train_step
 * with this rank's own B_local >= 1 transitions.  Rank r computes its per-sample rows, continues the Float64 running sum
 * rank r - 1 published (rank 0 starts from 0) with its rows in sample order and publishes the sum and the running sample
 * count; every rank then applies the final sum of rank world - 1 with B = the chained count.  So after every update every
 * rank holds the same θ, acc, g and loss, and they equal snk_qnet_train_step on the ranks' minibatches concatenated in rank
 * order, bit for bit, for any world (world = 1 is snk_qnet_train_step).  Ranks wait for each other on the device (flags over
 * peer memory, no host synchronisation); a wait that gives up after ~20 s sets the flag snk_qnet_group_status_host reports.
 * Every rank must call train_step the same number of times.  A rank keeps all B_local rows resident: B_local x 0.73 MB of
 * device memory, plus 2.9 MB of peer memory.
 * Set-up, once: create -> export_host (64 bytes) -> [the host language moves every rank's 64 bytes to every rank: MPI,
 * Distributed.jl, torch.distributed, a file ...] -> connect_host(world x 64 bytes in rank order, own entry ignored).
 * connect_local wires the groups of ONE process (virtual ranks on one GPU, each driven from its own stream).  The Q-net must
 * outlive its group. */
#define SNK_QNET_GROUP_HANDLE_BYTES 64
typedef struct snk_qnet_group_s *snk_qnet_group;
SNK_API int snk_qnet_group_create(snk_qnet_group *out, snk_qnet q, int world, int rank);
SNK_API int snk_qnet_group_destroy(snk_qnet_group g);
SNK_API int snk_qnet_group_export_host(snk_qnet_group g, uint8_t *handle64);
SNK_API int snk_qnet_group_connect_host(snk_qnet_group g, const uint8_t *handles_world_x_64, int n_handles);
SNK_API int snk_qnet_group_connect_local(snk_qnet_group g, const snk_qnet_group *peers, int n_peers);
SNK_API int snk_qnet_group_train_step(snk_qnet_group g, const float *states, const uint8_t *actions, const double *targets,
                                      int64_t B_local, float *acc, double eta, double rho, double epsilon, float *grad_out,
                                      float *loss_out, void *cuda_stream);
/* SNK_ERR_TIMEOUT if a wait gave up on a peer (synchronises) */
SNK_API int snk_qnet_group_status_host(snk_qnet_group g, int *timed_out);
/* profiling aid (SNK_QNET_BF16): device buffer of 512 int64 that receives clock64 stamps of the conv phases of CTA 0 on every
 * later forward (64 slots for each of its first 8 iterations, tools/qnet_phases17.py); NULL switches it off */
SNK_API int snk_qnet_debug_timing(snk_qnet q, long long *device_buf);

/* ---- Laplace deviation matrix  compute_D.jl:9-31, 66-81; la_utils.jl:14-36, 154-169 -------- */
/* D is P x K Float64, column-major (column k = snapshot k).  Welford mean / M2 over the columns in
 * column order, var = M2 / max(K-1,1), then D .-= mean, all in Float64 without FMA contraction so
 * the result is bit-identical to the Julia loop.  mean/var (P) may be NULL. */
SNK_API int snk_center_columns(double *D, int64_t P, int64_t K, double *mean, double *var, void *cuda_stream);
/* deviation_matrix[:, position] = Float64.(theta)  (compute_D.jl:67-71): theta = Flux.destructure(q_net) as Float32 on the
 * device, position 0-based. */
/* sample_model (la_utils.jl:83-95): w = mean + sqrt.(|var|) .* z1 / sqrt(2) + D * z2 / sqrt(2(K-1)), all Float64 on the
 * device; z1 (P) and z2 (K) are the injected standard-normal draws (rand(MvNormal(0, I))). */
SNK_API int snk_laplace_sample_weights(const double *mean, const double *var, const double *D, int64_t P, int64_t K,
                                       const double *z1, const double *z2, double *w, void *cuda_stream);
SNK_API int snk_d_store_snapshot(double *D, int64_t P, int64_t K, int64_t position, const float *theta, void *cuda_stream);

/* ---- Gram of the deviation matrix  plot_traj.jl:10-16 (svd(D), S.^2/(K-1) = eig(D'D)/(K-1)) ------------
 * G = A A^T with A = D^T: A is K x P row-major (row k = snapshot k) — byte-identical to Julia's P x K
 * column-major deviation_matrix.  G is K x K Float32 row-major (symmetric).
 *   snk_gram_pack  splits A (Float64 or Float32) into bf16 hi and lo planes inside the workspace;
 *   snk_gram       runs the tcgen05 kernel (TMA loads, TMEM accumulators) + the deterministic split-K
 *                  reduction.  terms = 1: hi hi^T (bf16 inputs, ~3 digits); terms = 3: hi hi^T + hi lo^T + lo hi^T
 *                  (~2^-17 relative per product), all three into one accumulator.  Only the tiles that meet the upper
 *                  triangle are computed; the reduction mirrors them, so G is exactly symmetric.
 *   block_k: 32 or 64 (0 = default); splits: split-K factor (0 = fill the SMs); the same `splits` must be
 *   given to snk_gram_workspace_bytes. */
#define SNK_DTYPE_F32 1
#define SNK_DTYPE_F64 2
SNK_API int snk_gram_workspace_bytes(int64_t K, int64_t P, int splits, size_t *bytes);
/* tile engine: 2 (default) = CTA pairs sharing 256x256 tiles (tcgen05 cta_group::2), 1 = single-CTA 128x256 tiles */
SNK_API int snk_gram_config(int cta_group);
SNK_API int snk_gram_pack(const void *A, int a_dtype, int64_t P, int64_t K, void *workspace, void *cuda_stream);
SNK_API int snk_gram(const void *workspace, int64_t P, int64_t K, int terms, int block_k, int splits, float *G,
                     void *cuda_stream);

/* ---- block-wise pieces, for the row-sharded multi-GPU Gram (SURVEY 8e: rank g owns rows_g of A) -----------
 * planes: bf16 [rows][pitch] arrays hi and lo (snk_gram_planes_layout gives bytes per plane and the pitch).
 * snk_gram_block:  Y (rows_a x rows_b, ld ldY) = hi_a hi_b^T [+ hi_a lo_b^T + lo_a hi_b^T]: a finished block of G; the b
 *                  planes may be a local copy of a peer's planes.  symmetric != 0 (same planes on both sides): only the
 *                  tiles meeting the upper triangle are computed, the rest is mirrored.  scratch:
 *                  snk_gram_block_scratch_bytes.  snk_gram_block_flops: what the tensor pipe executes for such a block
 *                  (computed tiles, padded, x products) — the numerator of an MMA-rate figure.
 * snk_gram_transpose_block: G_block (rows_a x rows_b) = YT^T where YT is the (rows_b x rows_a) block ANOTHER rank
 *                  computed; YT may be a peer-memory pointer (the kernel reads it with plain loads over NVLink). */
SNK_API int snk_gram_planes_layout(int64_t rows, int64_t P, size_t *plane_bytes, int64_t *pitch_elems);
SNK_API int snk_gram_pack_planes(const void *A, int a_dtype, int64_t P, int64_t rows, void *hi, void *lo, void *cuda_stream);
SNK_API int snk_gram_block_scratch_bytes(int64_t rows_a, int64_t rows_b, int64_t P, int splits, size_t *bytes);
SNK_API int snk_gram_block(const void *a_hi, const void *a_lo, int64_t rows_a, const void *b_hi, const void *b_lo, int64_t rows_b,
                           int64_t P, int terms, int symmetric, int block_k, int splits, void *scratch, float *Y, int64_t ldY,
                           void *cuda_stream);
SNK_API int snk_gram_block_flops(int64_t rows_a, int64_t rows_b, int64_t P, int terms, int symmetric, double *executed);
SNK_API int snk_gram_transpose_block(const float *YT, int64_t ldYT, int64_t rows_a, int64_t rows_b, float *G, int64_t ldG,
                                     void *cuda_stream);
/* ---- the row-sharded Gram as ONE call per rank (one process per GPU; SURVEY 8b `snk_gram(..., comm)`, BASELINE config 5b)
 * rows_all[world]: rows of A owned by every rank; this rank owns rows_all[rank] rows x P.  Set-up, once:
 *   create -> export_host (192 bytes) -> [the host language moves the 192 bytes of every rank to every rank: MPI,
 *   Distributed.jl, torch.distributed, a file ...] -> connect_host(all handles, world x 192 bytes, own entry ignored).
 * snk_gram_shard_run(g, A_rows, ...) then enqueues the whole Gram on `cuda_stream`: pack -> planes ring over NVLink peer
 * memory under the tcgen05 main loop (G is symmetric: a rank multiplies its rows against its own and the next world/2
 * ranks' rows only) -> the other blocks are read, transposed, out of the memory of the peers that computed them; the phases
 * are separated by a device-side barrier over peer memory (no host synchronisation, no communicator).  Every rank must call
 * it the same number of times.  G_rows: (rows x K_total) Float32, leading dimension ldG >= K_total.  A_rows == NULL: the
 * planes (snk_gram_shard_planes) were already written by a producer (snk_qnet_sample_grads).
 * pack / ring / mirror / barrier are the phases on their own; connect_local wires shards of ONE process together
 * (virtual ranks on one GPU, used by the tests) — there the caller orders the phases itself. */
#define SNK_GRAM_SHARD_HANDLE_BYTES 192
typedef struct snk_gram_shard_s *snk_gram_shard;
SNK_API int snk_gram_shard_create(snk_gram_shard *out, const int64_t *rows_all, int world, int rank, int64_t P, int splits,
                                  int device);
SNK_API int snk_gram_shard_destroy(snk_gram_shard g);
SNK_API int snk_gram_shard_export_host(snk_gram_shard g, uint8_t *handle192);
SNK_API int snk_gram_shard_connect_host(snk_gram_shard g, const uint8_t *handles_world_x_192);
SNK_API int snk_gram_shard_connect_local(snk_gram_shard g, const snk_gram_shard *peers);
SNK_API int snk_gram_shard_run(snk_gram_shard g, const void *A_rows, int a_dtype, int terms, int block_k, float *G_rows,
                               int64_t ldG, void *cuda_stream);
SNK_API int snk_gram_shard_pack(snk_gram_shard g, const void *A_rows, int a_dtype, void *cuda_stream);
SNK_API int snk_gram_shard_ring(snk_gram_shard g, int terms, int block_k, void *cuda_stream);
SNK_API int snk_gram_shard_mirror(snk_gram_shard g, float *G_rows, int64_t ldG, void *cuda_stream);
/* which blocks rank `rank` of `world` computes in the ring (the rest are mirrored): for step i = 0 .. *steps-1 the peer is
 * (rank + i) % world; a0/a1[i] = the range of its OWN rows it multiplies, b0/b1[i] = the range of the peer's rows (the last
 * step of an even world is shared: the lower rank takes the first rows of its own block against all of the peer's, the
 * higher rank all of its own against the remaining rows of the peer's).  Arrays of world/2 + 1 entries.  Pure arithmetic. */
SNK_API int snk_gram_shard_schedule(const int64_t *rows_all, int world, int rank, int *steps, int64_t *a0, int64_t *a1, int64_t *b0,
                                    int64_t *b1);
SNK_API int snk_gram_shard_barrier(snk_gram_shard g, void *cuda_stream);
SNK_API int snk_gram_shard_planes(snk_gram_shard g, void **hi, void **lo, int64_t *pitch_elems);
/* SNK_ERR_TIMEOUT if a barrier gave up waiting for a peer (synchronises) */
SNK_API int snk_gram_shard_status_host(snk_gram_shard g, int *timed_out);

/* device memory that other ranks of the box can map (cudaIpc*): allocate, export a 64-byte handle, import a
 * peer's handle, copy (works on peer-mapped pointers: the planes ring of the sharded Gram) */
SNK_API int snk_ipc_alloc(void **p, size_t bytes);
SNK_API int snk_ipc_free(void *p);
SNK_API int snk_ipc_export(void *p, uint8_t *handle64);
SNK_API int snk_ipc_import(const uint8_t *handle64, void **p);
SNK_API int snk_ipc_close(void *p);
SNK_API int snk_copy_async(void *dst, const void *src, size_t bytes, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* SNAKE_B200_H */
