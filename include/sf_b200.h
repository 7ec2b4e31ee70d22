/* sf_b200.h — C-ABI of the B200-native batched Space Fortress simulator.
 *
 * Drop-in boundary for ONE path of agakshat/spacefortress: env step + observation render +
 * auto-reset. Each entry point names the reference interface it replaces (paths are relative
 * to the reference repository root):
 *
 *   reference (CPython type `_spacefortress.Game`, python/spacefortress/src/pymodule.cpp)
 *   -------------------------------------------------------------------------------------
 *   Game(config, lw, grayscale, width, height, viewport)   pymodule.cpp:319-354  -> sf_create
 *   tp_dealloc                                              pymodule.cpp:295-302  -> sf_destroy
 *   press_key / release_key / step_one_tick(ms) / draw()    pymodule.cpp:199-247  -> sf_step (one call per batch)
 *   is_game_over()                                          pymodule.cpp:233-240  -> done[] of sf_step
 *   new Game per episode (ssf_env.py:163-178)               -> sf_reset / auto-reset inside sf_step
 *   pb_pixels + cv2 gray + cv2.resize (ssf_env.py:205, rl/envs.py:29) -> obs[] of sf_step / sf_render
 *   37 read-only getters (pymodule.cpp:372-411), dump()     -> sf_get_state (+ host formatting)
 *   (no setters exist: pymodule.cpp:48-74 commented out)    -> sf_set_state (teacher forcing)
 *   SubprocVecEnv.step/reset (gym_vecenv 1.0, rl/train.py:32,60,80) -> sf_step / sf_step_host / sf_rollout
 *   sum(info) / final_rewards bookkeeping (rl/train.py:81-88)       -> sf_episode_stats
 *
 * Conventions: plain C types only; every function returns an int status (SF_OK == 0) and never
 * calls exit() (the reference does on a bad config key, config.cpp:35-38); sf_last_error() gives
 * the message of the last failure on the calling thread. Pointers named d_* are DEVICE pointers
 * on the handle's GPU, h_* are HOST pointers. `stream` is a cudaStream_t passed as void*
 * (NULL = the legacy default stream). Device-pointer calls are asynchronous on `stream` and do
 * not synchronise the host. There is no CPU fallback: without a CUDA device sf_create fails. */
#ifndef SF_B200_H
#define SF_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SF_OK 0
#define SF_ERR_INVALID 1  /* bad argument (unknown game type, null pointer, size mismatch) */
#define SF_ERR_CUDA 2     /* a CUDA runtime call failed; see sf_last_error() */
#define SF_ERR_UNSUPPORTED 3

#define SF_MAX_MISSILES 20 /* pymodule.cpp:472, game.hh:3 */
#define SF_MAX_SHELLS 20   /* pymodule.cpp:473, game.hh:4 (the device keeps 4 slots: <= 3 shells can be alive) */
#define SF_NUM_STATS 13    /* game.hh:29-43 */
#define SF_OBS_H 84        /* rl/envs.py:29 */
#define SF_OBS_W 84
#define SF_NATIVE_H 92     /* int(460*.2), ssf_env.py:58 */
#define SF_NATIVE_W 90     /* int(450*.2), ssf_env.py:57 */
#define SF_NUM_EPISODE_STATS 24

/* key mask bits per step: the env sends FIRE, THRUST[, LEFT, RIGHT] every step (ssf_env.py:213-229) */
enum { SF_KEY_FIRE = 1, SF_KEY_THRUST = 2, SF_KEY_LEFT = 4, SF_KEY_RIGHT = 8 };

/* per-step event bits (replace the event strings of game.cpp:124-127 and Collisions, game.hh:45-47) */
enum {
  SF_EV_MISSILE_FIRED = 1 << 0, SF_EV_FORTRESS_FIRED = 1 << 1, SF_EV_HIT_FORTRESS = 1 << 2,
  SF_EV_VLNER_INCREASED = 1 << 3, SF_EV_VLNER_RESET = 1 << 4, SF_EV_FORTRESS_DESTROYED = 1 << 5,
  SF_EV_HIT_DEAD_FORTRESS = 1 << 6, SF_EV_EXPLODE_BIGHEX = 1 << 7, SF_EV_EXPLODE_SMALLHEX = 1 << 8,
  SF_EV_SHELL_HIT_SHIP = 1 << 9, SF_EV_SHIP_RESPAWN = 1 << 10, SF_EV_FORTRESS_RESPAWN = 1 << 11,
  SF_EV_COL_BIGHEX = 1 << 12, SF_EV_COL_SMALLHEX = 1 << 13, SF_EV_COL_MISSILE_FORTRESS = 1 << 14,
  SF_EV_COL_SHELL_SHIP = 1 << 15,
  SF_EV_PRESS_FIRE = 1 << 16, SF_EV_PRESS_THRUST = 1 << 17, SF_EV_PRESS_LEFT = 1 << 18, SF_EV_PRESS_RIGHT = 1 << 19,
  SF_EV_MISSED_SHOT = 1 << 20,
  SF_EV_EPISODE_RESET = 1 << 21, /* the env was auto-reset after this step */
  SF_EV_STICKY = 1 << 22         /* sticky actions: a tick of this agent step kept the held keys (sf_set_sticky_actions) */
};

/* sf_step / sf_rollout flags */
enum {
  SF_FLAG_RENDER = 1,       /* write the 84x84 observation */
  SF_FLAG_NO_AUTORESET = 2, /* leave finished envs finished (single-env facade: SSF_Env has no auto-reset) */
  SF_FLAG_ACTIONS_ARE_KEYMASKS = 4, /* actions[] already hold key masks instead of action ids */
  SF_FLAG_NATIVE_OBS = 8,   /* obs is the native 92x90 frame (SSF_Env.step) instead of 84x84 */
  SF_FLAG_RAW_REWARD = 16,  /* reward = Game.step_one_tick's int (pymodule.cpp:230): no Python-layer shaping, prev_vlner untouched */
  SF_FLAG_HOST_DELTA = 32   /* sf_step_host only: h_obs is page-locked and unchanged since the previous call (see sf_step_host) */
};

/* observation types of SSF_Env (ssf_env.py:51): the image is sf_step's d_obs; the other three are sf_features of the
 * current state, or the per-step rows of sf_rollout_features / sf_step_host_features */
enum { SF_OBS_IMAGE = 0, SF_OBS_FEATURES = 1, SF_OBS_NORMALIZED_FEATURES = 2, SF_OBS_MONITORS = 3 };

/* Per-env state record for get/set (teacher forcing, checkpointing, getters). Same members as the
 * reference's public Game fields (game.hh:84-107) + prev_vlner (ssf_env.py:92) + rand() position. */
typedef struct sf_state_record {
  double ship_x, ship_y, ship_vx, ship_vy, ship_angle;
  double fortress_angle, fortress_last_angle;
  double missile_x[SF_MAX_MISSILES], missile_y[SF_MAX_MISSILES];
  double missile_vx[SF_MAX_MISSILES], missile_vy[SF_MAX_MISSILES], missile_angle[SF_MAX_MISSILES];
  double shell_x[SF_MAX_SHELLS], shell_y[SF_MAX_SHELLS];
  double shell_vx[SF_MAX_SHELLS], shell_vy[SF_MAX_SHELLS], shell_angle[SF_MAX_SHELLS];
  float points, raw_points;
  uint32_t missile_mask, shell_mask;
  int32_t ship_alive, fortress_alive;
  int32_t ship_death_timer, fire_timer, thrust_timer, left_timer, right_timer;
  int32_t thrust_flag, fire_flag, left_flag, right_flag, turn_flag;
  int32_t fortress_timer, fortress_death_timer, fortress_vuln_timer;
  int32_t vulnerability, tick, time;
  int32_t stats[SF_NUM_STATS];
  int32_t prev_vlner;
  uint32_t rng_seed, rng_count;
  int32_t ep_return; /* running shaped return of the current episode (episode-stat bookkeeping) */
} sf_state_record;

typedef struct sf_handle sf_handle;

const char* sf_last_error(void);
int sf_version(void);

/* gametype: "youturn" | "autoturn" | "test-youturn" | "test-autoturn" (pymodule.cpp:331-343; unknown ->
 * SF_ERR_INVALID, the reference raises RuntimeError). action_set: 1 | 0 | -1 (ssf_env.py:65-90).
 * Allocates the SoA state slab for n_envs on CUDA device `device`. Envs are not yet reset. */
int sf_create(const char* gametype, int action_set, int n_envs, int device, sf_handle** out);
int sf_destroy(sf_handle* h);
int sf_num_envs(const sf_handle* h);
int sf_num_actions(const sf_handle* h);
int sf_action_keymask(const sf_handle* h, int action); /* -1 if out of range */
long long sf_state_bytes(const sf_handle* h);          /* device bytes held per handle */

/* (Re)seed the per-env libc-rand() streams (glibc TYPE_3, game.cpp:137-148). h_seeds==NULL: every env
 * gets seed 1 — the reference never calls srand, and forked gym_vecenv workers all replay that stream.
 * first_global_env offsets nothing in the seeds; it only labels this slab for the synthetic action hash
 * so that results are shard-invariant across GPUs. */
int sf_seed(sf_handle* h, const uint32_t* h_seeds, long long first_global_env, void* stream);

/* Extension for BASELINE.json configs[4] (auto-reset under episode-length variance): episode i continues from
 * tick h_ticks[i] (Game::mTick; mTime = 34 * tick, game.cpp:425-427), everything else is untouched. The
 * reference has fixed episodes of 5295 ticks (game.cpp:487-489); staggering the clocks makes the envs of a
 * batch finish at different steps. Same effect as sf_get_state / edit tick and time / sf_set_state. */
int sf_set_ticks(sf_handle* h, const int32_t* h_ticks);

/* SSF_Env.__init__/reset for all envs (d_mask==NULL) or for envs with d_mask[i]!=0: new Game
 * (game.cpp:18-82); prev_vlner is cleared only when clear_prev_vlner!=0 (= __init__, ssf_env.py:92).
 * d_obs (may be NULL) receives the first frame, layout per flags. */
int sf_reset(sf_handle* h, const uint8_t* d_mask, int clear_prev_vlner, uint8_t* d_obs, int flags, void* stream);

/* One SSF_Env.step for every env (ssf_env.py:208-253) + gym_vecenv auto-reset: actions -> key events ->
 * Game::stepOneTick(34) -> reward shaping -> done -> (reset) -> frame. Outputs may be NULL.
 *   d_actions int32[n]; d_obs uint8[n][84][84] (or [n][92][90] with SF_FLAG_NATIVE_OBS);
 *   d_reward int32[n] (the reference returns Python ints); d_done uint8[n]; d_fortkill uint8[n]
 *   (the reference's `info`, a bool: ssf_env.py:233,250); d_events uint32[n]. */
int sf_step(sf_handle* h, const int32_t* d_actions, uint8_t* d_obs, int32_t* d_reward, uint8_t* d_done,
            uint8_t* d_fortkill, uint32_t* d_events, int flags, void* stream);

/* T consecutive steps in ONE launch (state never leaves the SM between steps). d_actions int32[T][n],
 * or NULL for the synthetic policy: action = hash(action_seed, global_env, t) % num_actions (the same
 * stream sf_synthetic_action() gives on the host). Outputs are time-major: d_obs[T][n][84][84],
 * d_reward[T][n], d_done[T][n], d_fortkill[T][n]; any may be NULL. */
int sf_rollout(sf_handle* h, int T, const int32_t* d_actions, uint32_t action_seed, long long t0, uint8_t* d_obs,
               int32_t* d_reward, uint8_t* d_done, uint8_t* d_fortkill, int flags, void* stream);
int sf_synthetic_action(uint32_t action_seed, long long global_env, long long t, int num_actions);

/* Extension: action repeat (gym `frameskip`, EnvPool `frame_skip`, the MaxAndSkip wrapper without the max). With repeat
 * k, one agent step of an env with action a is what this loop around SSF_Env gives inside the gym_vecenv worker:
 *     R = 0; kill = False; ev = 0
 *     for j in range(k):
 *         obs, r, done, kill_j = env.step(a)     # key events, stepOneTick(34), shaping, prev_vlner: per tick as always
 *         R += r; kill |= kill_j; ev |= events_j
 *         if done: break                         # the repeat stops on the tick the episode ends
 *     (auto-reset at that tick)
 * reward = the int32 sum of the executed ticks' rewards (raw rewards under SF_FLAG_RAW_REWARD); done and fort_kill = set
 * by any executed tick; events = the OR of their bits (SF_EV_EPISODE_RESET included). The observation (frame or feature
 * row) is that of the state after the agent step, the first state of the new episode after an auto-reset: bit for bit
 * what sf_render / sf_features (float32) return then. Under SF_FLAG_NO_AUTORESET the repeat stops at done as well and
 * the env stays finished. SF_FLAG_ACTIONS_ARE_KEYMASKS repeats the key mask. The synthetic stream is hash(action_seed,
 * global_env, t0 + t) with t the agent step: all k ticks of a step use the same action.
 * The setting belongs to the handle (default 1, which is the plain one-tick step) and applies to every later call of
 * sf_step, sf_rollout, sf_step_host, sf_rollout_features and sf_step_host_features, whose T counts agent steps.
 * sf_reset, sf_render, sf_features, the env blobs and sf_episode_stats do not depend on it (episode lengths stay in
 * ticks; a blob row does not hold it). k < 1 or k > SF_MAX_ACTION_REPEAT (one episode) -> SF_ERR_INVALID, setting
 * unchanged. sf_action_repeat returns the setting, -1 for a NULL handle. */
#define SF_MAX_ACTION_REPEAT 5295
int sf_set_action_repeat(sf_handle* h, int k);
int sf_action_repeat(const sf_handle* h);

/* Extension: sticky actions (ALE's repeat_action_probability, Machado et al. 2018; Gymnasium ALE v5 and EnvPool default
 * to 0.25). A handle setting (p, sticky_seed), default p = 0, which is the plain step bit for bit. With p > 0 every
 * executed tick of every env makes one draw before its key processing:
 *     u = hash(sticky_seed, global_env, ((uint64)rng_count << 32) | tick)
 * (written out: c = rng_count << 32 | (uint32)tick; z = global_env * 0x9E3779B97F4A7C15 ^ c * 0xC2B2AE3D27D4EB4F ^
 * (sticky_seed << 32 | 0x57) in uint64; z ^= z >> 30; z *= 0xBF58476D1CE4E5B9; z ^= z >> 27; z *= 0x94D049BB133111EB;
 * z ^= z >> 31; u = z >> 32: the synthetic action hash with 0x57 in place of its 0x5F)
 * with global_env = first_global_env + i (the label of the synthetic action stream) and rng_count / tick the env's
 * PRE-tick values (rand() calls consumed, Game::mTick; sf_state_record.rng_count / .tick). The previous keys stick iff
 * (uint64)u < llround(p * 2^32): p = 0 never sticks, p = 1 always does. If they stick, the tick runs with the key mask
 * the env already holds (the FIRE / THRUST / LEFT / RIGHT flags of the state), otherwise with the agent's key mask. Every
 * key is sent every tick, so a sticky tick is a tick without press or release edges; fire stays edge-triggered.
 * With action repeat k the draw happens on each of the up-to-k ticks: the switch to a new action is delayed by a
 * geometric number of ticks. After an auto-reset the new game holds no keys, so a sticky first tick of an episode is
 * "no keys" (ALE resets its previous action to NOOP). SF_EV_STICKY is set on an agent step when any of its executed ticks
 * drew "stick", even if the held keys equal the action's. SF_FLAG_ACTIONS_ARE_KEYMASKS, SF_FLAG_NO_AUTORESET,
 * SF_FLAG_RAW_REWARD and the synthetic stream work as before: the draw applies after the action became a key mask.
 * The draw is a function of the env's state, not a counter: (rng_count, tick) never repeats within an env's life (tick
 * rises within an episode and every new game consumes rand() calls) except after an explicit rewind (sf_seed,
 * sf_set_ticks, sf_set_state), where repeating a draw is intended. So there is no per-env sticky state and no blob
 * change: a restored env (sf_load_envs) continues with exactly the draws it would have made, given the same (p, seed,
 * first_global_env); a fork into another slot has another label and diverges; results do not depend on the sharding
 * over GPUs. The hash differs from the synthetic action hash: sticky_seed == action_seed gives uncorrelated draws.
 * The setting applies to sf_step, sf_rollout, sf_step_host, sf_rollout_features and sf_step_host_features; sf_reset,
 * sf_render, sf_features, the env blobs and sf_episode_stats do not depend on it. p not finite or outside [0, 1] ->
 * SF_ERR_INVALID, setting unchanged. sf_sticky_actions returns p, -1 for a NULL handle. sf_sticky_draw (host only, no
 * GPU needed) is the device's draw: 1 if the keys stick, 0 if not, -1 for a p outside [0, 1]. */
int sf_set_sticky_actions(sf_handle* h, double p, uint32_t seed);
double sf_sticky_actions(const sf_handle* h);
int sf_sticky_draw(uint32_t seed, long long global_env, uint32_t rng_count, int32_t tick, double p);

/* Render the current state without stepping (Game.draw + gray + resize). */
int sf_render(sf_handle* h, uint8_t* d_obs, int flags, void* stream);

/* Host-buffer path (numpy drop-in for rl/train.py:79-80): H2D actions, step, D2H results, synchronous. Copies go
 * straight from/to the caller's buffers (use sf_host_alloc for them). h_obs may be NULL. Runs on streams the handle
 * owns: the slab is stepped in slices of consecutive envs so that the kernel of one slice overlaps the device->host
 * copy of the previous one. Ordered after everything queued with stream == NULL; work queued on any OTHER stream for
 * this handle (sf_save_envs and sf_load_envs included) must have completed before the call (sf_set_ticks, sf_get_state
 * and sf_set_state synchronise the device themselves).
 * SF_FLAG_HOST_DELTA: the caller promises that h_obs is page-locked (sf_host_alloc / cudaHostAlloc / cudaHostRegister,
 * 16-byte aligned) and that nothing but sf_step_host of this handle has written to it since the previous call that
 * passed the same pointer with this flag (see sf_host_forget). The frames of consecutive steps differ in a few dozen
 * bytes per env, so the library keeps a device copy of the buffer's contents and writes only the 64-byte granules (host cache lines) that
 * changed, straight into h_obs from the GPU; the buffer holds exactly what the full copy would have produced (resets, auto-resets and device-path steps in between included:
 * the comparison is against the buffer's contents, not the env's history). The first call for a buffer sends whole
 * frames. Fails with SF_ERR_INVALID if h_obs is not page-locked. */
int sf_step_host(sf_handle* h, const int32_t* h_actions, uint8_t* h_obs, int32_t* h_reward, uint8_t* h_done,
                 uint8_t* h_fortkill, uint32_t* h_events, int flags);
/* The library remembers the contents of up to 4 host buffers per handle (a caller may rotate a few; the least recently
 * used one is forgotten first). Before a buffer that was passed with SF_FLAG_HOST_DELTA is freed or reused for
 * something else, tell the library (h_obs == NULL: all of them); sf_destroy forgets everything. */
int sf_host_forget(sf_handle* h, const void* h_obs);
/* out3[0] = observation bytes the SF_FLAG_HOST_DELTA calls have written to host buffers, out3[1] = number of such calls,
 * out3[2] = number of rendering sf_step_host calls that sent whole frames. */
int sf_host_delta_stats(sf_handle* h, unsigned long long* out3);

/* Page-locked host memory for the buffers handed to sf_step_host: the device<->host copies then run as
 * direct DMA into the caller's arrays (pageable memory also works, but is staged by the driver). */
int sf_host_alloc(void** out, long long bytes);
int sf_host_free(void* p);

/* State records, host side (synchronous). first..first+count-1. */
int sf_get_state(sf_handle* h, int first, int count, sf_state_record* h_out);
int sf_set_state(sf_handle* h, int first, int count, const sf_state_record* h_in);

/* Env blobs: one env's complete game state as one fixed-size row, written and read on the device (checkpoint and resume,
 * forking an env into many slots, moving envs between handles or GPUs). Byte layout of a row (little endian):
 *     0  header: uint32 SF_ENV_BLOB_MAGIC, uint32 SF_ENV_BLOB_VERSION, uint32 gametype (0 youturn, 1 autoturn,
 *        2 test-youturn, 3 test-autoturn), uint32 0
 *    16  ship pos (double x, y), vel (double vx, vy)
 *    48  q0..q3 (int4 each: core word, live-slot mask, timers, points, tick, running episode return, prev_vlner)
 *   112  st0..st3 (int4 each: the 13 Stats counters, rand() ring index, rand() calls consumed, seed)
 *   176  missile pos[20] (double x, y)           496  shell pos[4], 560 shell vel[4] (double x, y)
 *   624  shell angle[4] (double)                 656  missile angle[20] (int16, degrees)
 *   696  rand() ring[31] (uint32)                820  zero up to SF_ENV_BLOB_BYTES
 * Rows are canonical: dead missile and shell slots and all padding are zero, so two envs in the same state give
 * byte-identical rows. Not in a row: the render caches (memos: a load invalidates them), the per-handle episode-stat
 * accumulators and the handle's first_global_env label. */
#define SF_ENV_BLOB_BYTES 832
#define SF_ENV_BLOB_VERSION 1
#define SF_ENV_BLOB_MAGIC 0x42465353u /* "SSFB" */
/* Row k of d_blob <- env d_env_idx[k] (d_env_idx == NULL: envs 0..count-1). An index outside [0, n) gives an all-zero
 * row (which a load rejects). d_blob is 16-byte aligned. Asynchronous on `stream`. */
int sf_save_envs(sf_handle* h, const int32_t* d_env_idx, int count, uint8_t* d_blob, void* stream);
/* Env d_env_idx[k] <- row k of d_blob (d_env_idx == NULL: envs 0..count-1). Rows with a bad header (magic, version or a
 * gametype other than the handle's) or a target index outside [0, n) are skipped and added to *d_rejected (int32,
 * device, may be NULL). Target indices must not repeat within one call; the same row may be loaded into many envs.
 * The loaded envs' render caches are invalidated. d_blob is 16-byte aligned. Asynchronous on `stream`. */
int sf_load_envs(sf_handle* h, const uint8_t* d_blob, const int32_t* d_env_idx, int count, int32_t* d_rejected, void* stream);

/* Finished-episode statistics accumulated on the device since the last call with reset!=0:
 * int64[SF_NUM_EPISODE_STATS] = {episodes, sum_return, sum_return^2, sum_length, sum of the 13 Stats
 * counters (game.hh:29-43; maxVlner summed), sum (int)points, sum round(raw_points*1000), sum fort_kills,
 * max maxVlner, steps, 2 reserved}. d_out is a device pointer (feed it to ncclAllReduce / torch.distributed);
 * integer sums make the reduction bitwise shard-invariant. */
int sf_episode_stats(sf_handle* h, long long* d_out, int reset, void* stream);

/* Consumer-side helper for the on-device rollout (rl/train.py:51-56,92-97: current_obs frame stack, zeroed on done,
 * scaled by 1/255 in rl/networks.py:35): the 4-frame stack of every env as the policy's first-layer input.
 * d_frames points at the OLDEST of 4 consecutive time-major frames [4][n][84][84] u8 (frame_stride_bytes apart);
 * d_valid[i] = frames since env i's last reset, capped at 4 (older frames read as 0). d_out is bf16
 * [n][21][21][64], i.e. an NHWC tensor of shape (n, 64, 21, 21) in channels_last: channel = frame*16 + (y%4)*4 + (x%4)
 * of pixel (4*Y + y%4, 4*X + x%4) -- the space-to-depth form in which conv(4->16, k8, s4) is a 2x2 convolution
 * over 64 channels (same sums). value = bf16(u8 / 255). No handle: a pure function of its arguments. */
int sf_policy_input(const uint8_t* d_frames, long long frame_stride_bytes, int n, const int32_t* d_valid, void* d_out_bf16, void* stream);
/* the same with fp32 output for an fp32 / TF32 policy: value = fp32(u8) * fp32(1 / 255), bit for bit what torch's CUDA
 * `obs / 255.0` (rl/networks.py:43) computes (it multiplies by the reciprocal of the scalar) */
int sf_policy_input_f32(const uint8_t* d_frames, long long frame_stride_bytes, int n, const int32_t* d_valid, float* d_out_f32, void* stream);

/* Feature observations of the CURRENT state (SSF_Env._get_features, ssf_env.py:95-157), one row per env:
 * SF_OBS_FEATURES / SF_OBS_NORMALIZED_FEATURES: 15 + 4 key timers (youturn) or + 2 (autoturn) columns, SF_OBS_MONITORS: 10.
 * vdir / aim / ndist are Game::computeExtra (game.cpp:282-312, including its fdist bug) evaluated in fp64 on the device;
 * before the first tick of an episode they are 0 (the reference's mExtra is uninitialised there). len(shells) counts
 * shells and the vulnerability timer is the real one (the reference's getters for them are broken: pymodule.cpp:44-45,
 * 131-134). d_out: float32 (sf_features) or float64 (sf_features_f64, what np.array(f) holds in the reference)
 * [n][sf_num_features]. */
int sf_num_features(const sf_handle* h, int obs_type);
int sf_features(sf_handle* h, int obs_type, float* d_out, void* stream);
int sf_features_f64(sf_handle* h, int obs_type, double* d_out, void* stream);

/* Feature observations as outputs of the step (render off), from the state-only kernel that steps the envs: no second
 * launch, and no frames. Row t of an env is bit for bit what sf_features (float32) returns after tick t: the state after
 * the tick, the first state of the new episode after an auto-reset, the finished state under SF_FLAG_NO_AUTORESET.
 * obs_type: SF_OBS_FEATURES, SF_OBS_NORMALIZED_FEATURES or SF_OBS_MONITORS. SF_FLAG_RENDER, SF_FLAG_NATIVE_OBS,
 * SF_FLAG_HOST_DELTA, a bad obs_type or a NULL features pointer -> SF_ERR_INVALID.
 * sf_rollout_features: T consecutive steps in ONE launch with feature observations instead of frames. d_features float32
 * [T][n][sf_num_features(h, obs_type)], row t = the features after tick t (auto-reset included); the other outputs as in
 * sf_rollout plus d_events [T][n] (any may be NULL); d_actions NULL = the synthetic stream. T <= 0 -> SF_ERR_INVALID. */
int sf_rollout_features(sf_handle* h, int obs_type, int T, const int32_t* d_actions, uint32_t action_seed, long long t0,
                        float* d_features, int32_t* d_reward, uint8_t* d_done, uint8_t* d_fortkill, uint32_t* d_events,
                        int flags, void* stream);
/* sf_step_host with feature rows [n][F] into h_features. If h_features is page-locked, the kernel writes the rows in place
 * through its device alias, like the small per-env arrays; otherwise a device buffer is copied back. Same ordering rules
 * as sf_step_host. */
int sf_step_host_features(sf_handle* h, int obs_type, const int32_t* h_actions, float* h_features, int32_t* h_reward,
                          uint8_t* h_done, uint8_t* h_fortkill, uint32_t* h_events, int flags);

/* Score digits (drawScore, draw.cpp:160-173) are font dependent: the reference asks fontconfig for "monospace" bold and
 * draws whatever face the machine has. The built-in digits are a 7-segment face on the same metrics. Where a real cairo and
 * the deployment's font exist, tools/dump_cairo_glyphs.py renders the masks and this call installs them: h_alpha
 * [10][5 * 27] = coverage of digit d drawn in every one of the 7 slots, over native rows 1..5 x columns 32..58;
 * h_slot[27] = the slot (0..6) that owns a strip column, 255 for none. Both NULL: back to the built-in face. Rebuilds the
 * static tables (default observation, pre-resampled chunks) and uploads them; synchronises the device. */
int sf_set_glyph_masks(sf_handle* h, const uint8_t* h_alpha, const uint8_t* h_slot);

/* Static tables built at sf_create (host copies, for tests/inspection): background frames. */
int sf_background(const sf_handle* h, uint8_t* h_native /*[92*90]*/, uint8_t* h_obs /*[84*84]*/);

/* Host-only (no GPU needed): compose the static layers of a frame from the same tables the kernels use
 * (background hexagons, fortress sprite or fortress explosion, score digits, vulnerability bar) into a
 * native 92x90 frame. Used by the CPU test-suite to check the table builder. fortress_alive < 0, points < 0
 * or vulnerability < 0 leave that layer out (all three: the bare background). */
int sf_host_static_frame(int fortress_alive, int fortress_angle_deg, int points, int vulnerability, int kill_bar,
                         uint8_t* h_native /*[92*90]*/, uint8_t* h_bg_obs /*[84*84] or NULL*/);

#ifdef __cplusplus
}
#endif
#endif /* SF_B200_H */
