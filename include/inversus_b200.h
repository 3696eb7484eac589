/*
 * inversus_b200.h -- C ABI of the B200-native batched INVERSUS simulator.
 *
 * This is the drop-in boundary for the reference's rollout hot path. The reference
 * (Jason-Hoford/inversus-reinforcement-learning) is pure Python and has no FFI; the interface
 * being replaced is the duck type of `MultiEnvRunner` (inversus_rl/env_wrappers.py:447-528) as
 * the trainer consumes it (inversus_rl/training.py:76,99,124,149 and :220,261,292,317).
 * Each entry point below cites the reference code it stands in for. Signatures carry only plain
 * pointers, sizes and scalars: no torch types. INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - Every function returns an inv_status code (0 = INV_OK); inv_last_error() gives the text of
 *     the calling thread's last failure.
 *   - There is no CPU fallback: every compute entry point fails with INV_ERR_NO_DEVICE unless its
 *     device (the handle's; the current one for handle-free calls) is an sm_100 part. The scratch-size
 *     queries (inv_ln_relu_partials, inv_encode_partials_floats, inv_conv3x3_wgrad_scratch_floats) and
 *     the inv_host_* calls run anywhere.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream). Calls enqueue
 *     work and return; nothing synchronises unless stated. One handle per GPU; a handle is not
 *     thread-safe.
 *   - The board is the reference's default 15 x 10 (inversus/config.py:7-8). Tiles: bit = 1 is
 *     WHITE. Directions and action ids follow env_wrappers.py:24-37 (UP, RIGHT, DOWN, LEFT).
 *   - Device buffers returned by inv_get_buffer are owned by the handle and stay valid until
 *     inv_destroy; their contents are overwritten by the next reset/step.
 */
#ifndef INVERSUS_B200_H
#define INVERSUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INV_ABI_VERSION 1

#define INV_BOARD_W 15
#define INV_BOARD_H 10
#define INV_OBS_CHANNELS 12
#define INV_OBS_ELEMS (INV_OBS_CHANNELS * INV_BOARD_H * INV_BOARD_W) /* 1800 */
#define INV_EXTRA_ELEMS 4
#define INV_MAX_BULLETS 16
#define INV_NUM_ACTIONS 13
#define INV_PACKED_STATE_BYTES 80 /* 5 x 16 B planes per env (DESIGN.md "state layout") */

/* draw-table mode: per env per call, INV_TABLE_STRIDE u32; the scripted opponent's draws start
 * at 0, (auto-)reset draws at INV_TABLE_RESET_OFF */
#define INV_TABLE_STRIDE 64
#define INV_TABLE_RESET_OFF 16
#define INV_STREAM_RESET 0xFFFFFFFFu
/* the third counter word of seat 0's draws in inv_scripted_actions is INV_STREAM_SEAT0 | step_count
 * (step_count < 2^31): a range no simulator stream (step_count, INV_STREAM_RESET) can reach */
#define INV_STREAM_SEAT0 0x80000000u

typedef enum {
    INV_OK = 0,
    INV_ERR_INVALID_ARG = -1,
    INV_ERR_CUDA = -2,
    INV_ERR_INVALID_ACTION = -3, /* ValueError of discrete_to_action, env_wrappers.py:66 */
    INV_ERR_BULLET_OVERFLOW = -4,
    INV_ERR_NOT_RESET = -5,
    INV_ERR_NO_DEVICE = -6
} inv_status;

typedef enum { INV_MODE_DUMMY = 0, INV_MODE_SELFPLAY = 1 } inv_mode;         /* env_wrappers.py:305-316 */
typedef enum { INV_DIFFICULTY_EASY = 0, INV_DIFFICULTY_HARD = 1 } inv_difficulty; /* env_wrappers.py:81-89 */
/* INV_OBS_NONE: no observation tensor at all (the extra vector and every other output are still
 * written). For consumers that read the packed state directly -- the PPO trainer's policy does,
 * through inv_encode_fwd -- the step then moves about 200 bytes per env instead of 3.8-7.4 KB. */
typedef enum { INV_OBS_F32 = 0, INV_OBS_BF16 = 1, INV_OBS_U8 = 2, INV_OBS_NONE = 3 } inv_obs_dtype;

/* inv_config.flags */
#define INV_FLAG_AUTO_RESET 1u /* fuse the trainer's reset-on-done (training.py:140-151) into step */
#define INV_FLAG_P2_VIEW 2u    /* also emit the P2-perspective observation (selfplay, env_wrappers.py:311) */
#define INV_FLAG_REWARD_F64 4u /* also keep the step reward as the binary64 sum the reference returns from
                                  SingleInversusRLEnv.step (env_wrappers.py:343-444), before its float32 cast */

/* bits of the per-env info byte (env_wrappers.py:360-427) */
#define INV_INFO_LANDED_HIT 1u
#define INV_INFO_GOT_HIT 2u
#define INV_INFO_WIN 4u
#define INV_INFO_LOSE 8u

/* sticky device status bits (inv_poll_status) */
#define INV_STATUS_INVALID_ACTION 1u
#define INV_STATUS_BULLET_OVERFLOW 2u
#define INV_STATUS_BAD_INDEX 4u /* inv_reset_envs saw an index outside [0, n_envs): that entry was skipped */

typedef struct inv_sim inv_sim;

/* Mirrors MultiEnvRunner.__init__ (env_wrappers.py:450-469) plus the sharding/RNG knobs. */
typedef struct {
    int64_t n_envs;            /* envs owned by this handle (this rank's shard) */
    int64_t env_id_base;       /* global id of env 0: RNG is keyed by global id, so results do not depend on the shard count */
    uint64_t seed;             /* Philox key */
    int32_t mode;              /* inv_mode */
    int32_t difficulty;        /* inv_difficulty */
    int32_t max_episode_steps; /* env_wrappers.py:263 (trainer passes 500) */
    int32_t device;            /* CUDA device ordinal */
    int32_t obs_dtype;         /* inv_obs_dtype; F32 is the reference's layout (env_wrappers.py:190) */
    uint32_t flags;            /* INV_FLAG_* */
} inv_config;

/* Canonical unpacked state of one env: the parity surface (inv_export_state / inv_import_state).
 * Mirrors InversusEnv's fields (core.py:36-51) + SingleInversusRLEnv's (env_wrappers.py:261-270). */
typedef struct {
    uint32_t tiles[5];  /* bit (y*15+x): 1 = WHITE, 0 = BLACK */
    int32_t p1[5];      /* x, y, ammo, reload_counter, alive (game_types.py:53-63) */
    int32_t p2[5];
    int32_t n_bullets;
    int8_t bullets[INV_MAX_BULLETS][4]; /* x, y, dir, owner(0=P1,1=P2), in list order (core.py:51) */
    int32_t step_count; /* env_wrappers.py:265 */
    uint32_t episode;   /* resets so far - 1 (RNG counter word); 0xFFFFFFFF before the first reset */
    double episode_return; /* env_wrappers.py:266 */
} inv_env_state;

typedef enum {
    INV_BUF_OBS_P1 = 0,     /* [n,12,10,15] obs_dtype   -- grid tensor, env_wrappers.py:190-235 */
    INV_BUF_EXTRA_P1 = 1,   /* [n,4] f32                -- extra vector, env_wrappers.py:238-243 */
    INV_BUF_OBS_P2 = 2,     /* as above from P2's view (INV_FLAG_P2_VIEW) */
    INV_BUF_EXTRA_P2 = 3,
    INV_BUF_REWARD = 4,     /* [n] f32   -- env_wrappers.py:525 */
    INV_BUF_DONE = 5,       /* [n] u8    -- env_wrappers.py:526 */
    INV_BUF_INFO = 6,       /* [n] u8    -- INV_INFO_* bits */
    INV_BUF_EPISODE_STEPS = 7,  /* [n] i32 -- info["episode_steps"], env_wrappers.py:441 */
    INV_BUF_EPISODE_RETURN = 8, /* [n] f64 -- info["episode_return"], env_wrappers.py:442 */
    INV_BUF_PACKED_STATE = 9,   /* [5,n] uint4 planes, INV_PACKED_STATE_BYTES per env */
    INV_BUF_DEBUG_RESULT = 10,  /* [n] u8 -- return value of the last inv_debug_phase call */
    INV_BUF_REWARD_F64 = 11     /* [n] f64 -- the unrounded reward (INV_FLAG_REWARD_F64) */
} inv_buffer;

/* engine calls reachable one at a time through inv_debug_phase (parity tests only) */
typedef enum {
    INV_PHASE_TRY_MOVE = 0,     /* core.py:249  try_move_player(dir=arg, pid) */
    INV_PHASE_SPAWN_BULLET = 1, /* core.py:298  spawn_bullet(dir=arg, pid) */
    INV_PHASE_WIDE_SHOT = 2,    /* core.py:328  spawn_wide_shot(pid, dir=arg) */
    INV_PHASE_RELOAD = 3,       /* core.py:383  _reload_ammo() */
    INV_PHASE_UPDATE_BULLETS = 4, /* core.py:399 update_bullets() */
    INV_PHASE_STEP_PLAYERS = 5, /* core.py:497  step_players(a1=arg, a2=arg2) */
    INV_PHASE_ENGINE_RESET = 6, /* core.py:55   reset() */
    INV_PHASE_DUMMY_POLICY = 7  /* env_wrappers.py:69 dummy_opponent_policy -> action id in the result byte */
} inv_phase;

int inv_abi_version(void);
const char *inv_last_error(void);
int inv_device_count(void);

/* MultiEnvRunner(num_envs, opponent_type, difficulty, max_episode_steps, seed)  env_wrappers.py:450 */
int inv_create(const inv_config *cfg, inv_sim **out);
int inv_destroy(inv_sim *sim);
int inv_get_config(const inv_sim *sim, inv_config *out);

/* MultiEnvRunner.reset()  env_wrappers.py:471-483 : starts a new episode in every env and
 * writes the observations. */
int inv_reset(inv_sim *sim, void *stream);

/* MultiEnvRunner.envs[i].reset() for i in idx (training.py:149): idx is a DEVICE array of
 * `count` local env indices (no duplicates). Rewrites those envs' observations only. */
int inv_reset_envs(inv_sim *sim, const int64_t *idx_dev, int64_t count, void *stream);

/* MultiEnvRunner.step(action_ids, opponent_policy)  env_wrappers.py:485-528.
 * a_p1_dev: [n] int8 action ids of P1. a_p2_dev: [n] int8 ids of P2 in selfplay mode (the
 * result of running opponent_policy on the P2 view of the previous step), NULL in dummy mode.
 * One fused kernel: P2's scripted action, engine tick, reward, done, optional auto-reset,
 * observation write-out. Ids outside 0..12 set INV_STATUS_INVALID_ACTION and act as NONE. */
int inv_step(inv_sim *sim, const int8_t *a_p1_dev, const int8_t *a_p2_dev, void *stream);

/* Same call with HOST buffers: copies the actions in, steps, copies every output out and
 * synchronises -- the literal numpy-in / numpy-out contract of MultiEnvRunner.step. Any output
 * pointer may be NULL to skip it. obs is [n,12,10,15] of the handle's obs dtype. Returns
 * INV_ERR_INVALID_ACTION (state untouched) if an id is outside 0..12, like the reference's
 * ValueError. */
int inv_step_host(inv_sim *sim, const int8_t *a_p1, const int8_t *a_p2, void *obs_p1, float *extra_p1,
                  void *obs_p2, float *extra_p2, float *reward, uint8_t *done, uint8_t *info,
                  int32_t *episode_steps, double *episode_return);
int inv_reset_host(inv_sim *sim, void *obs_p1, float *extra_p1, void *obs_p2, float *extra_p2);

/* One episode that ended in a step: what the trainer reads at training.py:140-151 (episode_return,
 * episode_steps, win) for the envs whose done flag is set. */
typedef struct {
    int64_t env;            /* local env index, ascending within a step */
    double episode_return;  /* info["episode_return"], env_wrappers.py:442 */
    int32_t episode_steps;  /* info["episode_steps"],  env_wrappers.py:441 */
    uint32_t info;          /* INV_INFO_* bits (win / lose / landed_hit / got_hit) */
} inv_episode_event;

/* The step as a trainer with a GPU-resident policy consumes it: actions come from host memory, the
 * observations -- grid and extra -- stay on the device (inv_get_buffer), reward / done / info arrive
 * dense (any may be NULL), and the episodes that ended in this step arrive as a compact list in env
 * order: *n_events records in events[0 .. capacity). 6 bytes per env plus 24 per finished episode
 * cross the bus instead of inv_step_host's 34 per env. capacity >= n_envs can never overflow; if
 * fewer fit, *n_events still holds the true count and INV_ERR_INVALID_ARG is returned (the step has
 * been taken). Same argument errors as inv_step_host. */
int inv_step_host_events(inv_sim *sim, const int8_t *a_p1, const int8_t *a_p2, float *reward, uint8_t *done,
                         uint8_t *info, inv_episode_event *events, int64_t capacity, int64_t *n_events);

/* How inv_step_host delivers float32 observations to host memory. nthreads = 0: one plain
 * device-to-host copy (PCIe-bound, about 7.2 KB per env). nthreads > 0 (default: the host's
 * hardware threads, at most 32): the kernel also emits each observation as its packed 1800-bit
 * row (256 B/env); the copy engine moves the float32 data of a fraction `dma_fraction` of the envs
 * while `nthreads` host threads expand the packed rows of the rest with non-temporal stores.
 * dma_fraction < 0 = keep balancing the two legs from their measured rates (default). Format
 * conversion only; other dtypes and batches under 4096 envs always use the plain copy. */
int inv_set_host_path(inv_sim *sim, int nthreads, double dma_fraction);
int inv_get_host_path(const inv_sim *sim, int *nthreads, double *dma_fraction, double *last_dma_s,
                      double *last_expand_s);

/* The host half of that path, usable on its own (no GPU involved): expand packed observation rows
 * bits[n][64] (u32; bit i of a row = observation element i, 1800 used) into dst[n][1800] f32 for
 * rows [first, first+count), on nthreads host threads (AVX-512 / AVX2 non-temporal stores). */
int inv_host_expand_f32(const uint32_t *bits, float *dst, int64_t first, int64_t count, int nthreads);

/* The id check of the *_host calls, usable on its own (no GPU involved): copies ids[n] to staged[n]
 * (staged may be ids itself) and returns INV_OK if every id is in 0..12, INV_ERR_INVALID_ACTION
 * otherwise -- the ValueError of discrete_to_action, env_wrappers.py:66. One AVX2 pass. */
int inv_host_stage_action_ids(const int8_t *ids, int8_t *staged, int64_t n);

/* page-locked host memory for the *_host calls (pageable memory works too, slower) */
int inv_host_alloc(void **out, int64_t nbytes);
int inv_host_free(void *p);

int inv_get_buffer(inv_sim *sim, int which, void **dev_ptr, int64_t *nbytes);

/* Draw source. table_dev = NULL (default): Philox4x32-10, counter (global env id, episode,
 * stream, k/4), key = seed. Otherwise the next reset/step reads draw k of env i from
 * table_dev[i*INV_TABLE_STRIDE + k] (see INV_TABLE_*): the "injected RNG draws" parity mode. */
int inv_set_draw_table(inv_sim *sim, const uint32_t *table_dev);

/* parity surface: canonical state out / in (synchronous, host buffers) */
int inv_export_state(inv_sim *sim, inv_env_state *out_host, int64_t first, int64_t count);
int inv_import_state(inv_sim *sim, const inv_env_state *in_host, int64_t first, int64_t count);

/* Resume from a snapshot: copy [5, n] uint4 planes (a copy of INV_BUF_PACKED_STATE taken earlier
 * from a handle with the same n_envs) into the handle. Together with the seed this restores the
 * whole simulation: every later draw is a pure function of (seed, global env id, episode,
 * step_count, k), all of which live in the packed state. The observation buffers are NOT
 * refreshed; call inv_obs_from_packed on the handle's own state (or step) to get them. */
int inv_load_packed_state(inv_sim *sim, const void *packed_dev, void *stream);

/* Rebuild observations from packed-state snapshots (build_observation, env_wrappers.py:173-245,
 * over data copied earlier from INV_BUF_PACKED_STATE): a PPO rollout keeps 80 B/env-step instead
 * of 7216 B and decodes minibatches on demand. packed_dev: [5, stride] uint4 planes, entries
 * [0,count) decoded; view 0 = P1, 1 = P2. */
int inv_obs_from_packed(inv_sim *sim, const void *packed_dev, int64_t stride, int64_t count, int view,
                        int obs_dtype, void *obs_out_dev, float *extra_out_dev, void *stream);

/* Test hook: run ONE engine method of core.py on every env (same device functions the fused
 * step kernel is built from). The per-env return value lands in INV_BUF_DEBUG_RESULT. */
int inv_debug_phase(inv_sim *sim, int phase, int pid, int arg, int arg2, void *stream);

/* synchronises `stream`, returns and clears the sticky INV_STATUS_* bits */
int inv_poll_status(inv_sim *sim, void *stream, uint32_t *bits);

/* PPOAgent.compute_advantages (inversus_rl/ppo_agent.py:127-157) over a device-resident rollout
 * laid out [T][N] (time-major, N envs): GAE per env, walking time backwards, float32 in the
 * reference's operation order. last_value_dev: [N] bootstrap values or NULL for 0 (the reference
 * always passes 0, ppo_agent.py:170). N = 1 with T = buffer length reproduces the reference's
 * flat-list behaviour bit for bit. Runs on the current device. */
int inv_gae(const float *reward_dev, const float *value_dev, const uint8_t *done_dev,
            const float *last_value_dev, double gamma, double lam, int32_t T, int64_t N, float *adv_dev,
            float *ret_dev, void *stream);

/* Fused (conv bias +) (residual +) LayerNorm + ReLU of the policy's channels-last bf16 path (the
 * memory-bound glue between the convolutions of inversus_rl/policies.py:27-45,94-100; the
 * contractions themselves stay in cuDNN/cuBLAS, run bias-free). A sample is D = H*W*C contiguous
 * bf16 values in HWC order, gamma/beta are [D] bf16 in the same order, cbias is the [C] bf16
 * per-channel convolution bias (may be NULL), statistics are fp32. res may be NULL.
 * D % C == 0, C % 8 == 0, 512 % (C/8) == 0, D <= 20480.
 *   fwd: y = relu(LN(x + cbias [+ res]) * gamma + beta); writes mean[B], rstd[B] for the backward.
 *   bwd: dx (also the gradient of res), dgamma[D], dbeta[D], dcbias[C] (fp32, dcbias may be NULL);
 *        partials is scratch of inv_ln_relu_partials(D) * (2*D + C) floats.
 * All pointers are device pointers on the current device. */
int inv_ln_relu_partials(int32_t D);
int inv_ln_relu_fwd(const void *x, const void *res, const void *cbias, const void *gamma, const void *beta,
                    int64_t B, int32_t D, int32_t C, float eps, void *y, float *mean, float *rstd, void *stream);
int inv_ln_relu_bwd(const void *dy, const void *x, const void *res, const void *cbias, const void *gamma,
                    const void *beta, const float *mean, const float *rstd, int64_t B, int32_t D, int32_t C,
                    void *dx, float *dgamma, float *dbeta, float *dcbias, float *partials, void *stream);

/* Layer 1 of the policy evaluated straight from packed env states (csrc/encoder_kernels.cu):
 *   y = relu(LayerNorm(conv1(build_observation(state)) + b1) * gamma + beta)
 * i.e. inversus_rl/policies.py:27-31,94 applied to the observation of env_wrappers.py:173-245,
 * without materialising the observation. packed_dev: [5, stride] uint4 planes (a copy or view of
 * INV_BUF_PACKED_STATE), entries [0, count); view 0 = P1, 1 = P2. w1: [32,12,3,3] fp32 (checkpoint
 * layout), b1: [32]; gamma_hwc / beta_hwc: LayerNorm affine permuted to [10,15,32] fp32.
 *   fwd: y_out [count,10,15,32] bf16 (channels-last), extra_out [count,4] f32 (the extra vector of
 *        env_wrappers.py:238-243; may be NULL), mean_out / rstd_out [count] f32 for the backward.
 *   bwd: dy [count,10,15,32] bf16 -> dw1 [32,12,3,3], db1 [32], dgamma_hwc / dbeta_hwc [4800], fp32.
 *        partials: scratch of inv_encode_partials_floats() floats. Deterministic (no atomics).
 * Pure functions of their arguments: no handle; they run on the current device. */
int inv_encode_partials_floats(void);
int inv_encode_fwd(const void *packed_dev, int64_t stride, int64_t count, int view, const float *w1, const float *b1,
                   const float *gamma_hwc, const float *beta_hwc, float eps, void *y_out, float *extra_out,
                   float *mean_out, float *rstd_out, void *stream);
int inv_encode_bwd(const void *packed_dev, int64_t stride, int64_t count, int view, const float *w1, const float *b1,
                   const float *gamma_hwc, const float *beta_hwc, const float *mean, const float *rstd, const void *dy,
                   float *dw1, float *db1, float *dgamma_hwc, float *dbeta_hwc, float *partials, void *stream);

/* Weight gradient of a 3x3, padding-1 convolution over the 15 x 10 board on the tcgen05 tensor cores
 * (csrc/wgrad_kernels.cu), for the policy's conv3 / conv4 (inversus_rl/policies.py:36-43):
 *   dw[co][ky][kx][ci] = sum over (n, y, x) of dy[n, y, x, co] * x[n, y + ky - 1, x + kx - 1, ci]
 * dy: [B,10,15,cout] bf16 and x: [B,10,15,cin] bf16, both channels-last and 16-byte aligned;
 * (cout, cin) = (128, 128), (128, 64) or (64, 32): conv4, conv3, conv2. dw: [cout][3][3][cin] fp32 (the
 * memory order of a channels-last filter). partials: scratch of
 * inv_conv3x3_wgrad_scratch_floats(cin, cout) floats. Deterministic. */
int64_t inv_conv3x3_wgrad_scratch_floats(int32_t cin, int32_t cout);
int inv_conv3x3_wgrad(const void *dy, const void *x, int64_t B, int32_t cin, int32_t cout, float *dw, float *partials,
                      void *stream);

/* Per-row transpose + fp32<->bf16 conversion: dst[r][b*A + a] = src[r][a*B + b], a < A, b < B, for
 * `rows` rows with leading dimensions ld_src / ld_dst (elements). Exactly one side is fp32, the
 * other bf16. Carries the head weight of policies.py:61-75 between the checkpoint's CHW column
 * order and the HWC order of channels-last activations (and the gradient back). */
int inv_transpose_cast(const void *src, int32_t src_is_f32, int64_t ld_src, void *dst, int32_t dst_is_f32,
                       int64_t ld_dst, int64_t rows, int32_t A, int32_t B, void *stream);

/* The evaluator's two device steps (csrc/eval_kernels.cu; DESIGN.md "evaluator"). Handle-free: one
 * launch on `stream` on the current device, capturable in a CUDA graph.
 * packed_dev / stride: [5, stride] uint4 planes (a view of INV_BUF_PACKED_STATE), entries [0, count).
 *
 * inv_select_actions: logits [count, 13] fp32 (contiguous rows) -> actions_out [count] int8.
 *   greedy != 0: the first index of the maximum (torch.argmax). greedy == 0: one Philox4x32-10 draw r,
 *   key = seed, counter = (gid_base + i, episode, step_count, 0x80000000 | seat), the env's pre-step
 *   counter words; inverse CDF in fp32: m = max, e_j = expf(l_j - m), S = e_0 + ... + e_12 in order,
 *   the smallest j with (r * 2^-32) * S < e_0 + ... + e_j, else the last j with e_j > 0. seat: 0 or 1.
 *   packed_dev may be NULL when greedy. A row holding NaN or +inf, or only -inf, gets id -1, which
 *   the next inv_step reports as INV_STATUS_INVALID_ACTION.
 *
 * inv_episode_tally: call after each inv_step of an auto-reset handle with its done / info /
 *   episode_steps / episode_return buffers and its post-step packed state. An env whose episode with
 *   index (episode - 1) ended in the step and whose index is < quota adds into its column of
 *   counts_dev int32 [4][count] (wins, losses, draws = done with neither INV_INFO_WIN nor
 *   INV_INFO_LOSE, sum of episode lengths) and return_sum_dev f64 [count] (summed in step order).
 *   remaining_dev (one int32) is zeroed and then receives the number of envs whose post-step
 *   episode is < quota. quota * max_episode_steps must be below 2^31. */
int inv_select_actions(const float *logits, int64_t count, const void *packed_dev, int64_t stride, int64_t gid_base,
                       uint64_t seed, int seat, int greedy, int8_t *actions_out, void *stream);
int inv_episode_tally(const uint8_t *done, const uint8_t *info, const int32_t *episode_steps,
                      const double *episode_return, const void *packed_dev, int64_t stride, int64_t count, int64_t quota,
                      int32_t max_episode_steps, int32_t *counts_dev, double *return_sum_dev, int32_t *remaining_dev,
                      void *stream);

/* inv_scripted_actions: the scripted dummy (env_wrappers.py:69-170) as a player of either seat, one
 *   int8 action id per env into actions_out [count], from the pre-step packed state (planes 0-2 of
 *   entries [0, count); csrc/eval_kernels.cu, DESIGN.md "evaluator"). Handle-free, one launch on
 *   `stream`, capturable in a CUDA graph, no synchronisation. difficulty: INV_DIFFICULTY_EASY / _HARD.
 *   seat 1 (P2): exactly the opponent of an INV_MODE_DUMMY step, drawing from counter
 *     (gid_base + i, episode, step_count, k/4), the stream that step consumes. A selfplay handle
 *     stepped with a_p2 = these ids reproduces a dummy-mode handle of the same seed, env ids and P1
 *     actions bit for bit.
 *   seat 0 (P1): the same rule with the roles exchanged: it chases / shoots at P2, steps only onto
 *     WHITE (P1's walkable colour) and returns 0 without a draw when P1 is dead; counter
 *     (gid_base + i, episode, INV_STREAM_SEAT0 | step_count, k/4).
 *   The fourth counter word k/4 < 16 keeps both apart from inv_select_actions (0x80000000 | seat).
 *   INV_ERR_INVALID_ARG: count < 0, NULL pointers, stride < count, seat or difficulty not 0/1,
 *   gid_base outside [0, 2^32 - count]. */
int inv_scripted_actions(const void *packed_dev, int64_t stride, int64_t count, int64_t gid_base, uint64_t seed,
                         int seat, int difficulty, int8_t *actions_out, void *stream);

/* kernel launches issued through this handle so far (bench.py's gpu_launches) */
int64_t inv_launch_count(const inv_sim *sim);

#ifdef __cplusplus
}
#endif
#endif /* INVERSUS_B200_H */
