// sf_kernels.cu — kernels and the C-ABI (include/sf_b200.h) of the B200-native batched Space Fortress
// simulator. sm_100a only; no CPU fallback: every entry point fails with SF_ERR_CUDA without a device.
//
// Kernels
//   sf_rollout_kernel           fused step + render + auto-reset for T consecutive ticks (T=1 == sf_step). One block
//                               of 24 warps per SM owns groups of <= 32 envs: warp 0 steps them one env per lane
//                               (SoA, 128-bit loads/stores) up to two ticks ahead and prepares the next stage, the
//                               other warps run the block-cooperative frame pipeline of sf_render.cuh and stream the
//                               84x84 frames to HBM.
//                               Groups beyond the first 148 are handed out first come first served (SfSched); between
//                               the ticks of a launch the group's scalars stay in shared memory (SfStepSmem); the static
//                               tables arrive as one bulk copy of a per-handle image (sf_pack_static_kernel).
//                               Three instantiations (SfRollMode): step, step with host delta (sf_step_host), and draw
//                               (sf_render, sf_reset: warp 0 loads the current state instead of stepping it).
//   sf_step_state_kernel        the state-only step (render off), one env per thread, T agent steps of up to k ticks of
//                               one action (sf_set_action_repeat). <FEAT, PLAIN, STICKY, FINAL>:
//                               FEAT: a feature row per env and agent step (sf_rollout_features, sf_step_host_features);
//                               PLAIN: one tick per agent step, no sticky actions, no final observations;
//                               STICKY: sticky actions (sf_set_sticky_actions, p > 0), at any k;
//                               FINAL = SF_FINAL_IN_KERNEL / SF_FINAL_DEFERRED: final observations (sf_set_final_obs).
//                               When frames need the split route (frames_need_split), each agent step is this kernel at
//                               T = 1 followed by a SF_ROLL_DRAW launch.
//   sf_final_reset_kernel       the deferred auto-reset of the envs whose final frames have just been drawn.
//   sf_features_kernel          the feature observation types of ssf_env.py:95-157 of the current state, one env per thread.
//   sf_policy_input_kernel      4-frame stack -> the policy's first-layer input (bf16 or fp32, space-to-depth NHWC).
//   sf_reset_kernel / sf_seed_kernel / sf_get_state_kernel / sf_set_state_kernel / sf_pack_static_kernel
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sf_b200.h"
#include "sf_geom.h"
#include "sf_render.cuh"
#include "sf_state.cuh"
#include "sf_step.cuh"
#include "sf_tables.h"

#define SF_BLOCK (32 * SF_RENDER_WARPS)  // sf_render.cuh: one block per SM

// ------------------------------------------------------------------------------------------------
// synthetic policy: stateless counter hash (SURVEY.md §8(d)); same function on host and device
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline unsigned sf_hash3(unsigned seed, unsigned long long env, unsigned long long t, unsigned salt = 0x5Fu) {
  unsigned long long z = (env * 0x9E3779B97F4A7C15ull) ^ (t * 0xC2B2AE3D27D4EB4Full) ^ ((unsigned long long)seed << 32 | salt);
  z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27; z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (unsigned)(z >> 32);
}
__host__ __device__ inline int sf_hash_action(unsigned seed, unsigned long long env, unsigned long long t, int num_actions) {
  return (int)(((unsigned long long)sf_hash3(seed, env, t) * (unsigned)num_actions) >> 32);
}
// Sticky actions (sf_set_sticky_actions): does the tick of env `env` whose pre-tick rand() count and tick are (rng_count,
// tick) keep the keys the env holds? threshold = llround(p * 2^32). Keyed on the env's state, not on a counter: the pair
// never repeats within an env's life, so a restored env makes the draws it would have made. Its own salt: with
// sticky_seed == action_seed the draws are not the synthetic actions' hash.
#define SF_STICKY_SALT 0x57u
__host__ __device__ inline bool sf_sticky_hash(unsigned seed, unsigned long long env, unsigned rng_count, int tick, unsigned long long threshold) {
  return (unsigned long long)sf_hash3(seed, env, (unsigned long long)rng_count << 32 | (unsigned)tick, SF_STICKY_SALT) < threshold;
}

// ------------------------------------------------------------------------------------------------
// finished-episode statistics: warp-reduced, then one atomic per field per warp
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ long long sf_warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Finished-episode statistics of the `finished` lanes of a warp (called by all 32 lanes). Out of line and by VALUE: a
// reference to the env's registers handed to a function that is not inlined forces the whole SfEnv into local memory in
// the caller (measured: the state-only kernel lost 30 %).
__device__ __noinline__ void sf_accumulate_episode_vals(unsigned long long* epi, bool finished, int lane, int ret_i, int length, int points_bits, int raw_bits,
                                                        int max_vlner, int4 st0, int4 st1, int4 st2) {
  long long f[SF_NUM_EPISODE_STATS];
  long long ret = ret_i;
  f[0] = 1; f[1] = ret; f[2] = ret * ret; f[3] = length;
  f[4] = st0.x; f[5] = st0.y; f[6] = st0.z; f[7] = st0.w;
  f[8] = st1.x; f[9] = st1.y; f[10] = st1.z; f[11] = st1.w;
  f[12] = st2.x; f[13] = st2.y; f[14] = st2.z; f[15] = st2.w; f[16] = max_vlner;
  f[17] = (long long)__float2int_rz(__int_as_float(points_bits));
  f[18] = __double2ll_rn((double)__int_as_float(raw_bits) * 1000.0);
  f[19] = st1.y;  // fortress kills of the episode (== destroyedFortresses; rl/train.py:81 sums info)
  f[20] = 0; f[21] = 0; f[22] = 0; f[23] = 0;
#pragma unroll
  for (int k = 0; k < 20; k++) {
    long long v = sf_warp_sum_ll(finished ? f[k] : 0);
    if (lane == 0 && v) atomicAdd(&epi[k], (unsigned long long)v);
  }
  int mv = finished ? max_vlner : 0;
  mv = sf_warp_max(mv);
  if (lane == 0 && mv) atomicMax(&epi[20], (unsigned long long)mv);
}
// the finished lanes' pending Stats increments go to the arrays first (reductions: read back through L2)
__device__ __forceinline__ void sf_accumulate_episode(const SfDev& D, int env, SfEnv& e, bool finished, int lane) {
  int4 st0 = make_int4(0, 0, 0, 0), st1 = st0, st2 = st0;
  if (finished) { sf_flush_stats(D, env, e); st0 = __ldcg(&D.st0[env]); st1 = __ldcg(&D.st1[env]); st2 = __ldcg(&D.st2[env]); }
  sf_accumulate_episode_vals(D.epi, finished, lane, e.q3.w, e.q3.z, e.q3.x, e.q3.y, e.st3.x, st0, st1, st2);
}

// the renderer's view of one stepped env (written by the env's lane into the block's record array)
__device__ __forceinline__ void sf_make_env_rec(const SfEnv& e, int env, unsigned shell_vis, SfEnvRec& r) {
  r.px = e.pos.x; r.py = e.pos.y;
  r.core = (unsigned)e.q0.x; r.pmask = (unsigned)e.q0.y;
  r.points_i = __float2int_rz(__int_as_float(e.q3.x));
  r.vuln = e.q1.z;
  r.kill_bar = (e.q1.z > 10 && e.q1.y < 250) ? 1 : 0;
  r.env = env;
  r.s0 = 0; r.ebox = 0;
  if (!(r.core & SF_CORE_SHIP_ALIVE)) {  // explosion sprite box (draw.cpp:235-237)
    const SfPt c = sf_xform_base(r.px, r.py);
    r.ebox = (((c.x >> 8) - 13) + 64) | ((((c.y >> 8) - 13) + 64) << 8);
  }
  r.life = (unsigned)e.st3.z + 1u;
  r.building = 0;  // decided by sf_publish_recs
  r.ns = sf_count_strokes(r.core, r.pmask, shell_vis);
  r.shell_vis = (int)shell_vis;
}

// Device-resident scheduling state of sf_rollout_kernel (one per handle; zero at creation, self re-arming): with more
// groups than blocks, the groups after the first gridDim.x are handed out first come first served (the groups differ
// in cost and the launch ends with the slowest block: +5..8 % at 65 536 envs over static striding).
// (Tried and dropped: dealing the envs of a one-group-per-block launch to the blocks by a cost key read from their
// state, so that every block gets the same mix of dead and live ships — the spread of the block times fell only from
// 9.8 % to 7.7 % and the sort at the end of every launch cost more than that gained.)
struct SfSched {
  int next_group, done;                 // groups handed out beyond the first gridDim.x; blocks that have finished
};

struct SfRollArgs {
  int T, EB, ngroups, flags;  // EB = envs per group (<= 32), ngroups = ceil(n / EB): set by group_shape
  const int* actions;  // [T][n] or NULL
  unsigned action_seed;
  long long t0;
  unsigned char* obs;  // [T][n][obs_bytes]
  int* reward;         // [T][n]
  unsigned char* done;
  unsigned char* fortkill;
  unsigned* events;
  SfSched* sched;      // NULL: static assignment (block b owns groups b, b + gridDim.x, ...; no hand-out); set by launch_fused / launch_draw
  int env0, envn;      // the envs this launch steps: [env0, env0 + envn) (sf_step_host steps the slab in slices)
  // SF_FLAG_HOST_DELTA (sf_step_host, T == 1): every block ends by sending the changed granules of its own frames
  uint4* host_obs;     // device alias of the caller's page-locked observation buffer, or NULL
  uint4* mirror;       // device copy of what that buffer holds
  unsigned long long* delta_stats;
  const unsigned char* draw_mask;  // SF_ROLL_DRAW: the envs to draw (NULL: all); the others' frames are not written
};
// The feature rows of sf_rollout_features / sf_step_host_features: float32 [T][n][cols], row t = the state after tick t. A
// parameter of the state-only kernel of its own: SfRollArgs is 128 bytes, and with these members appended the compiler
// gave the kernel without feature rows 80 registers instead of 72 (different code from the same source).
struct SfFeatArgs {
  float* out;      // NULL: no feature rows
  int kind, cols;  // SF_OBS_FEATURES / SF_OBS_NORMALIZED_FEATURES / SF_OBS_MONITORS, sf_feature_cols
};
// Sticky actions: a parameter of the state-only kernel of its own, for the same reason as SfFeatArgs
struct SfStickyArgs {
  unsigned long long threshold;  // llround(p * 2^32): 0 never sticks, 2^32 always
  unsigned seed;
};
// Final observations at auto-reset (sf_set_final_obs): a parameter of the state-only kernel of its own, like SfStickyArgs.
// SF_FINAL_IN_KERNEL: a finished env writes step[env] (and, with feature rows, its final row into rows) just before its
// new game. SF_FINAL_DEFERRED (T = 1 launches with frames): a finished env writes step[env], is left finished and is
// marked in `pending`; a masked draw and sf_final_reset_kernel follow.
enum SfFinalMode { SF_FINAL_OFF, SF_FINAL_IN_KERNEL, SF_FINAL_DEFERRED };
struct SfFinalArgs {
  int* step;               // [n]: the agent step whose events carry SF_EV_EPISODE_RESET (written only for envs that end)
  float* rows;             // [n][F.cols] or NULL: the final feature rows (SF_FINAL_IN_KERNEL with feature rows)
  unsigned char* pending;  // [n]: SF_FINAL_DEFERRED's marks, cleared by sf_final_reset_kernel
  int t0;                  // the agent step index of the launch's step 0
};
enum SfRollMode { SF_ROLL_STEP, SF_ROLL_STEP_HOST_DELTA, SF_ROLL_DRAW };
// ticks per group, for both roles of a launch: a draw is the one frame of the current state
template <int MODE>
__device__ __forceinline__ int sf_roll_ticks(const SfRollArgs& A) { return MODE == SF_ROLL_DRAW ? 1 : A.T; }

// the key mask of an env's action at step t: given actions or the synthetic stream
__device__ __forceinline__ int sf_step_keys(const SfDev& D, const SfRollArgs& A, int env, int t) {
  int a = A.actions ? A.actions[(size_t)t * D.n + env]
                    : sf_hash_action(A.action_seed, (unsigned long long)(D.first_global_env + env), (unsigned long long)(A.t0 + t), D.num_actions);
  return (A.flags & SF_FLAG_ACTIONS_ARE_KEYMASKS) ? (a & 15) : D.keymask_of_action[min(max(a, 0), D.num_actions - 1)];
}
// a step's outputs at index t
__device__ __forceinline__ void sf_store_step_out(const SfDev& D, const SfRollArgs& A, int env, int t, const SfStepOut& o) {
  size_t oi = (size_t)t * D.n + env;
  if (A.reward) A.reward[oi] = o.reward;
  if (A.done) A.done[oi] = o.done;
  if (A.fortkill) A.fortkill[oi] = o.fort_kill;
  if (A.events) A.events[oi] = o.events;
}

// ------------------------------------------------------------------------------------------------
// fused step + render
// ------------------------------------------------------------------------------------------------
// One block renders groups of EB envs (persistent over the groups it owns, group-major, T ticks each). Per tick:
// warp 0 steps the group (one env per lane: SoA 128-bit loads/stores) and publishes the env records; then all
// warps run the block-cooperative frame pipeline (sf_render.cuh).
// one tick of a group (warp 0, one env per lane): step, outputs, auto-reset, staged env record
__device__ __noinline__ void sf_step_group(const SfDev& D, const SfRollArgs& A, int group, int t, SfEnvRec* recs) {
  const int lane = threadIdx.x & 31;
  const SfHot* H = &sf_block_smem().hot;  // the step's tables from shared memory
  const bool autoreset = !(A.flags & SF_FLAG_NO_AUTORESET);
  const int env = A.env0 + group * A.EB + lane;
  const bool mine = lane < A.EB && env < A.env0 + A.envn;
  SfEnv e;
  bool finished = false;
  unsigned shell_vis = 0;
  SF_ST_BEGIN(__ballot_sync(0xffffffffu, mine));
  SfStepSmem& SS = sf_block_smem().step;
  const bool first_tick = t == 0, last_tick = t == A.T - 1;
  if (mine) {
    if (first_tick) sf_load_env(D, env, e);
    else {  // between the ticks of a launch the group's scalars live in shared memory
      e.pos = SS.pos[lane]; e.vel = SS.vel[lane];
      e.q0 = SS.q0[lane]; e.q1 = SS.q1[lane]; e.q2 = SS.q2[lane]; e.q3 = SS.q3[lane]; e.st3 = SS.st3[lane];
      e.d0 = SS.d0[lane]; e.d1 = SS.d1[lane]; e.d2 = SS.d2[lane];
    }
    SF_ST_USE(e.q0.x, e.q0.y);
    SF_ST(8);
    SfStepOut o;
    sf_env_step(D, H, env, e, sf_step_keys(D, A, env, t), autoreset, (A.flags & SF_FLAG_RAW_REWARD) != 0, o);
    sf_store_step_out(D, A, env, t, o);
    finished = o.done && autoreset;
    shell_vis = o.shell_vis;
  }
  SF_ST_RESTART(0xffffffffu);
  if (__any_sync(0xffffffffu, finished)) {
    sf_accumulate_episode(D, env, e, finished, lane);
    if (finished) { sf_new_game(D, H, env, e); shell_vis = 0; }  // gym_vecenv: the returned obs is the first frame of the new episode
  }
  if (mine) {
    if (last_tick) sf_store_env(D, env, e);
    else {
      SS.pos[lane] = e.pos; SS.vel[lane] = e.vel;
      SS.q0[lane] = e.q0; SS.q1[lane] = e.q1; SS.q2[lane] = e.q2; SS.q3[lane] = e.q3; SS.st3[lane] = e.st3;
      if ((t & 7) == 7) sf_flush_stats(D, env, e);  // the pending Stats increments are 8-bit fields: every 8 ticks is often enough (as in sf_step_state_kernel)
      SS.d0[lane] = e.d0; SS.d1[lane] = e.d1; SS.d2[lane] = e.d2;
    }
    sf_make_env_rec(e, env, shell_vis, recs[lane]);
  } else recs[lane].env = -1;
  __syncwarp();
  SF_ST(15);
}

// SF_ROLL_DRAW (Game.draw of the current state): the group's records without a step (warp 0, one env per lane)
__device__ __forceinline__ void sf_load_group(const SfDev& D, const SfRollArgs& A, int group, SfEnvRec* recs) {
  const int lane = threadIdx.x & 31;
  const int env = A.env0 + group * A.EB + lane;
  const bool mine = lane < A.EB && env < A.env0 + A.envn && (!A.draw_mask || A.draw_mask[env]);
  if (mine) {
    SfEnv e;
    sf_load_env(D, env, e);
    sf_make_env_rec(e, env, sf_visible_shells(D, env, (unsigned)e.q0.y), recs[lane]);
  } else recs[lane].env = -1;
  __syncwarp();
}

// The two roles of the rollout kernel, out of line (separate register allocations, see sf_stepper_ticks). Both walk the
// same sequence of groups: the block's first group is blockIdx.x, further ones are handed out first come first served
// (the groups differ in cost, and so do the SMs' speeds). Warp 0 fetches the id of the NEXT group when it starts a group
// and leaves it in shared memory (a ring indexed by the group count, SF_NEXT_GROUPS); the other warps read it when they
// are done with the current group, many barriers later. The steps of the next ticks (warp 0) run while the other warps
// draw the ticks before them, across groups too.
template <int MODE>
__device__ __forceinline__ void sf_stepper_role(const SfDev& D, const SfRollArgs& A) {
  const int lane = threadIdx.x & 31;
  SfBlockSmem& B = sf_block_smem();
  const bool native = (A.flags & SF_FLAG_NATIVE_OBS) != 0;
  int stage = 0, group = blockIdx.x;
#pragma unroll 1
  for (int k = 0; group < A.ngroups; k = (k + 1) % SF_NEXT_GROUPS) {
    if (lane == 0) B.next_group[k] = A.sched ? (int)gridDim.x + atomicAdd(&A.sched->next_group, 1) : group + (int)gridDim.x;
    sf_stepper_ticks(D, B, lane, native, sf_roll_ticks<MODE>(A), stage, [&](int t, SfStagePrep& Tm, int h) {
      if constexpr (MODE == SF_ROLL_DRAW) sf_load_group(D, A, group, Tm.env);
      else sf_step_group(D, A, group, t, &Tm.env[32 * h]);
    });
    group = B.next_group[k];
  }
  sf_stepper_drain(stage);
  // the last block to leave re-arms the counters for the next launch (every block has made its last fetch by then)
  if (lane == 0 && A.sched) {
    __threadfence();
    if (atomicAdd(&A.sched->done, 1) == (int)gridDim.x - 1) { A.sched->next_group = 0; A.sched->done = 0; __threadfence(); }
  }
}
// The step modes call the stepping warp's role out of line. The draw mode inlines it: its short preparation is all of
// warp 0's work, and out of line it reaches D and A through references to the kernel parameters (generic loads instead
// of constant-bank loads), which made a draw 1-2.5 % slower (DESIGN.md 4.1).
template <int MODE>
__device__ __noinline__ void sf_rollout_stepper(const SfDev& D, const SfRollArgs& A) { sf_stepper_role<MODE>(D, A); }

template <int MODE>
__device__ __forceinline__ void sf_rollout_drawer(const SfDev& D, const SfRollArgs& A) {
  const int lane = threadIdx.x & 31;
  SfBlockSmem& B = sf_block_smem();
  SfWarpSmem& W = sf_my_smem();
  SfFrameOut out;
  out.native = (A.flags & SF_FLAG_NATIVE_OBS) ? 1 : 0;
  out.obs_bytes = out.native ? (size_t)SF_NAT_H * SF_NAT_W : (size_t)84 * 84;
  out.obs = A.obs;
  out.tick_bytes = MODE == SF_ROLL_DRAW ? 0 : (size_t)D.n * out.obs_bytes;
  SfStageState st;
  st.stage = 0; st.prev_used = 0;
  int group = blockIdx.x;
#pragma unroll 1
  for (int k = 0; group < A.ngroups; k = (k + 1) % SF_NEXT_GROUPS) {
    sf_drawer_ticks(D, B, W, lane, out, sf_roll_ticks<MODE>(A), st);
    group = B.next_group[k];
  }
}

// ------------------------------------------------------------------------------------------------
// SF_FLAG_HOST_DELTA (sf_step_host). Between two steps of an env only a few dozen bytes of its frame change (the moving
// objects and now and then a score digit), so the frames are not copied: `mirror` is the device's copy of what the
// caller's page-locked buffer holds, the new frames are compared with it, and the granules that differ are stored
// straight into the host buffer (its device alias: posted writes across PCIe). The host buffer ends up identical to a
// full copy; the traffic is ~600-1100 B per env-step instead of 7056.
// ------------------------------------------------------------------------------------------------
// 64 bytes = a host cache line: the host's memory system sees no partial-line writes (with 8 ranks writing at once up to
// 19 % faster than 32-byte granules, DESIGN.md 7.4). A variant build may set 16 ... 256 bytes.
#ifndef SF_DELTA_GRANULE
#define SF_DELTA_GRANULE 64
#endif
#define SF_DELTA_LANES (SF_DELTA_GRANULE / 16)  // 16-byte chunks per granule: neighbouring lanes of one ballot
static_assert(SF_DELTA_GRANULE == 16 || SF_DELTA_GRANULE == 32 || SF_DELTA_GRANULE == 64 || SF_DELTA_GRANULE == 128 || SF_DELTA_GRANULE == 256,
              "SF_DELTA_GRANULE must be 16, 32, 64, 128 or 256 bytes (1 to 16 lanes of a warp's ballot)");

// The 16-byte chunks [c0, c1) of the frames, shared by `nthreads` threads (a multiple of 32) of which this is `tid`, with
// four loads in flight. The loop bound is the same for every lane, so whole warps take part in each ballot. Returns the
// chunks this thread sent.
__device__ __forceinline__ unsigned sf_host_delta_range(const uint4* cur, uint4* mirror, uint4* host, size_t c0, size_t c1, unsigned tid, unsigned nthreads) {
  const unsigned gsh = (threadIdx.x & 31) & ~(unsigned)(SF_DELTA_LANES - 1);
  unsigned sent = 0;
#pragma unroll 1
  for (size_t base = c0; base < c1; base += 4 * nthreads) {
    uint4 a[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const size_t i = base + u * nthreads + tid;
      a[u] = b[u] = make_uint4(0, 0, 0, 0);
      if (i < c1) { a[u] = __ldcg(cur + i); b[u] = __ldcg(mirror + i); }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const size_t i = base + u * nthreads + tid;
      const bool diff = (a[u].x != b[u].x) | (a[u].y != b[u].y) | (a[u].z != b[u].z) | (a[u].w != b[u].w);
      const unsigned m = __ballot_sync(0xffffffffu, diff);
      if (m == 0) continue;
      if (i < c1 && ((m >> gsh) & ((1u << SF_DELTA_LANES) - 1u))) { host[i] = a[u]; sent++; }  // whole granules
      if (diff) mirror[i] = a[u];
    }
  }
  return sent;
}

// stats[0] += the bytes the warp sent (one atomic per warp); stats[1] counts the calls
__device__ __forceinline__ void sf_host_delta_count(unsigned long long* stats, unsigned sent) {
  for (int o = 16; o; o >>= 1) sent += __shfl_xor_sync(0xffffffffu, sent, o);
  if ((threadIdx.x & 31) == 0 && sent) atomicAdd(&stats[0], (unsigned long long)sent * 16u);
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&stats[1], 1ull);
}

// Inside the step kernel: each block compares the frames of its own groups, still in L2. Blocks finish at different
// times (at T = 1 the median block is done after ~70 % of the launch), so most of this and most of the PCIe traffic
// hides under the slower blocks; a separate kernel would start after the slowest block (DESIGN.md 7.4: 110 -> 105 us).
__device__ __noinline__ void sf_block_host_delta(const SfDev& D, const SfRollArgs& A) {
  const size_t per16 = (size_t)(84 * 84) / 16;
  unsigned sent = 0;
#pragma unroll 1
  for (int group = blockIdx.x; group < A.ngroups; group += gridDim.x) {
    const int env_lo = A.env0 + group * A.EB, env_hi = min(env_lo + A.EB, A.env0 + A.envn);
    sent += sf_host_delta_range(reinterpret_cast<const uint4*>(A.obs), A.mirror, A.host_obs, (size_t)env_lo * per16, (size_t)env_hi * per16,
                                threadIdx.x, SF_BLOCK);
  }
  sf_host_delta_count(A.delta_stats, sent);
}

// The separate kernel, over the whole buffer: the only one for frames that are not a multiple of 16 bytes (native 92x90,
// 8280 B per env). The last (bytes % 16) bytes go every time.
__global__ void __launch_bounds__(256) sf_host_delta_kernel(const uint4* __restrict__ cur, uint4* __restrict__ mirror, uint4* __restrict__ host,
                                                            size_t n16, int tail, unsigned long long* stats) {
  const unsigned sent = sf_host_delta_range(cur, mirror, host, 0, n16, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
  if (tail && blockIdx.x == 0 && threadIdx.x < (unsigned)tail) {
    const size_t o = n16 * 16 + threadIdx.x;
    const unsigned char v = reinterpret_cast<const unsigned char*>(cur)[o];
    reinterpret_cast<unsigned char*>(host)[o] = v; reinterpret_cast<unsigned char*>(mirror)[o] = v;
  }
  sf_host_delta_count(stats, sent);
}

// (SF_ROLL_STEP_HOST_DELTA is a separate instantiation, used by sf_step_host only: the register allocation of the plain
// kernel is sensitive to anything that is added to its body, see DESIGN.md 7b. SF_ROLL_DRAW runs T = 1 with static groups.)
template <int MODE>
__global__ void __launch_bounds__(SF_BLOCK, 1) sf_rollout_kernel(const __grid_constant__ SfDev D, const __grid_constant__ SfRollArgs A) {
  sf_block_smem_init(D.static_image);
  sf_warp_smem_init(sf_my_smem(), threadIdx.x & 31);
  if (threadIdx.x < 32) {
    if constexpr (MODE == SF_ROLL_DRAW) sf_stepper_role<MODE>(D, A);
    else sf_rollout_stepper<MODE>(D, A);
  } else sf_rollout_drawer<MODE>(D, A);
  if (MODE == SF_ROLL_STEP_HOST_DELTA) {
    __syncthreads();  // every frame of this block's groups is written (the bulk copies were waited for before the patches)
    sf_block_host_delta(D, A);
  }
}

// once per handle (and after sf_set_glyph_masks): the static part of SfBlockSmem, built from the tables, as an image in
// global memory that the rendering kernels fetch with one bulk copy
__global__ void __launch_bounds__(SF_BLOCK) sf_pack_static_kernel(SfDev D, unsigned char* image) {
  sf_block_smem_fill(D.tab);
  __syncthreads();
  const int4* src = reinterpret_cast<const int4*>(&sf_block_smem());
  for (int k = threadIdx.x; k < (int)(SF_STATIC_BYTES / 16); k += blockDim.x) reinterpret_cast<int4*>(image)[k] = src[k];
}

// For a state that was not reached by stepping the env (new seed, forced record, loaded blob). The env's render caches
// (explosion sprite, resampled box) are keyed by the ship's life: the rand() calls consumed at its spawn + 1. That key
// names a life only along one rand() stream followed step by step: after a new seed the counter restarts, and a forced or
// loaded state may place a dead ship anywhere at a count that a life of this env's old state also had.
__device__ __forceinline__ void sf_forget_render_caches(const SfDev& D, int env) {
  D.expstamp[env] = 0;
  D.expo_meta[env] = make_uint2(0u, 0u);
}

__global__ void sf_seed_kernel(SfDev D, const unsigned* seeds) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= D.n) return;
  SfEnv e;
  sf_load_env(D, env, e);
  sf_srand(D, env, e, seeds ? seeds[env] : 1u);
  sf_forget_render_caches(D, env);
  sf_store_env(D, env, e);
}

__global__ void sf_set_ticks_kernel(SfDev D, const int* ticks) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= D.n) return;
  int4 q = D.q3[env];
  q.z = max(ticks[env], 0);
  D.q3[env] = q;
}

__global__ void sf_reset_kernel(SfDev D, const unsigned char* mask, int clear_prev_vlner) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= D.n) return;
  if (mask && !mask[env]) return;
  SfEnv e;
  sf_load_env(D, env, e);
  if (clear_prev_vlner) e.q1.w = 0;
  sf_new_game(D, &D.tab->hot, env, e);
  sf_store_env(D, env, e);
}


// ------------------------------------------------------------------------------------------------
// feature observations (ssf_env.py:95-157), one thread per env: of the current state (sf_features_kernel) or of the
// state after every agent step (sf_step_state_kernel<true, ...>)
// ------------------------------------------------------------------------------------------------
// columns of a row: 15 + the key timers (4 youturn, 2 autoturn) for features / normalized-features, 10 for monitors
__host__ __device__ inline int sf_feature_cols(int autoturn, int kind) { return kind == SF_OBS_MONITORS ? 10 : 15 + (autoturn ? 2 : 4); }

// computeExtra (game.cpp:282-312). The reference evaluates it inside updateShip while the ship is alive and keeps the
// values while it is dead; position, velocity and heading are frozen while dead, so evaluating it from the current
// state gives the same numbers. Before the first tick of a Game the reference's mExtra is uninitialised memory; the
// test harness zero-fills the Game, and so does this (tick 0 -> 0, 0, 0). fdist keeps the bug of the reference (Q11:
// the y term is ship.y - ship.y).
struct SfExtra { double vdir, aim, ndist; };
__device__ __forceinline__ SfExtra sf_compute_extra(const SfEnv& e) {
  SfExtra x;
  x.vdir = 0.0; x.aim = 0.0; x.ndist = 0.0;
  if (e.q3.z == 0) return x;
  const double ang = (double)((unsigned)e.q0.x & SF_CORE_ANGLE_MASK);
  if (SF_DSQRT(SF_DADD(SF_DMUL(e.vel.x, e.vel.x), SF_DMUL(e.vel.y, e.vel.y))) != 0.0) {   // Vector::norm (vector.cpp:30-32)
    const double o = atan2(-SF_DSUB(SF_FORT_Y, e.pos.y), SF_DSUB(SF_FORT_X, e.pos.x));
    const double v = atan2(e.vel.y, e.vel.x);
    double d = SF_DSUB(v, o);
    if (d > SF_PI) d = SF_DSUB(d, SF_PI * 2);
    if (d < -SF_PI) d = SF_DADD(d, SF_PI * 2);
    x.vdir = sf_rad2deg(d);
  }
  double o = atan2(SF_DSUB(e.pos.y, SF_FORT_Y), SF_DSUB(e.pos.x, SF_FORT_X));
  o = SF_DADD(SF_DSUB(sf_rad2deg(o), ang), 180.0);
  if (o < -180.0) o = SF_DADD(o, 360.0);
  x.aim = o;
  const double dx = SF_DSUB(e.pos.x, SF_FORT_X), dy0 = SF_DSUB(e.pos.y, e.pos.y);
  const double fdist = SF_DSQRT(SF_DADD(SF_DMUL(dx, dx), SF_DMUL(dy0, dy0)));
  x.ndist = SF_DADD(-1.0, SF_DDIV(SF_DSUB(fdist, 40.0), SF_DDIV(SF_DSUB(200.0, 40.0), 2.0)));   // normDist (game.cpp:282-284)
  return x;
}
__device__ __forceinline__ double sf_clip1(double v) { return v < -1.0 ? -1.0 : (v > 1.0 ? 1.0 : v); }
__device__ __forceinline__ double sf_pymod360(double v) {  // Python's float `v % 360`
  double m = fmod(v, 360.0);
  if (m != 0.0) { if (m < 0.0) m = SF_DADD(m, 360.0); } else m = 0.0;
  return m;
}

// The one definition of a feature row: o[0 .. sf_feature_cols) <- the observation `kind` of state e. Inline: it reads the
// env's registers through a reference (see sf_accumulate_episode_vals). Each value is stored as soon as it is computed,
// so the stepping kernel holds no row of doubles.
template <class OutT>
__device__ __forceinline__ void sf_feature_row(const SfEnv& e, bool autoturn, int kind, OutT* o) {
  const SfExtra x = sf_compute_extra(e);
  const unsigned core = (unsigned)e.q0.x;
  const double alive = (core & SF_CORE_SHIP_ALIVE) ? 1.0 : 0.0, falive = (core & SF_CORE_FORT_ALIVE) ? 1.0 : 0.0;
  const int vuln = e.q1.z;
  const double kill_window = (vuln > 10 && e.q1.y < 250) ? 1.0 : 0.0;   // vulnerability_timer < fortressVulnerabilityTime
  const int nm = __popc((unsigned)e.q0.y & SF_PMASK_MISSILES), ns = __popc(((unsigned)e.q0.y >> SF_PMASK_SHELL_SHIFT) & 0xFu);
  const double fang = 10.0 * (double)((core >> SF_CORE_FANG_SHIFT) & 63u), sang = (double)(core & SF_CORE_ANGLE_MASK);
  if (kind == SF_OBS_MONITORS) {          // ssf_env.py:96-108
    auto put = [&](int k, bool on) { o[k] = (OutT)(on ? 0.5 : -0.5); };
    put(0, nm > 0); put(1, falive != 0.0); put(2, vuln > 10); put(3, kill_window != 0.0);
    put(4, x.aim < 3); put(5, x.aim > 3);
    put(6, x.ndist > .75); put(7, x.ndist > .25); put(8, x.ndist < -.25); put(9, x.ndist < -.75);
  } else if (kind == SF_OBS_NORMALIZED_FEATURES) {  // ssf_env.py:109-133 (sic: max(vulnerability, 10)); np.clip(f, -1, 1)
    auto put = [&](int k, double v) { o[k] = (OutT)sf_clip1(v); };
    put(0, alive); put(1, SF_DDIV(e.pos.x, 90.0)); put(2, SF_DDIV(e.pos.y, 92.0)); put(3, SF_DDIV(e.vel.x, 10.0)); put(4, SF_DDIV(e.vel.y, 10.0));
    put(5, SF_DDIV(sang, 360.0)); put(6, SF_DDIV(x.aim, 180.0)); put(7, SF_DDIV(sf_pymod360(x.vdir), 360.0)); put(8, x.ndist);
    put(9, falive); put(10, SF_DDIV(fang, 360.0)); put(11, SF_DDIV((double)max(vuln, 10), 10.0)); put(12, kill_window);
    put(13, SF_DDIV((double)nm, 20.0)); put(14, SF_DDIV((double)ns, 20.0));
    const double max_ticks = 5294.0;  // np.floor(180000 / 34), ssf_env.py:166
    put(15, SF_DDIV((double)e.q2.x, max_ticks)); put(16, SF_DDIV((double)e.q2.y, max_ticks));
    if (!autoturn) { put(17, SF_DDIV((double)e.q2.z, max_ticks)); put(18, SF_DDIV((double)e.q2.w, max_ticks)); }
  } else {                               // 'features', ssf_env.py:134-157
    auto put = [&](int k, double v) { o[k] = (OutT)v; };
    put(0, alive); put(1, e.pos.x); put(2, e.pos.y); put(3, e.vel.x); put(4, e.vel.y); put(5, sang); put(6, x.aim); put(7, x.vdir); put(8, x.ndist);
    put(9, falive); put(10, fang); put(11, (double)vuln); put(12, kill_window); put(13, (double)nm); put(14, (double)ns);
    put(15, (double)e.q2.x); put(16, (double)e.q2.y);
    if (!autoturn) { put(17, (double)e.q2.z); put(18, (double)e.q2.w); }
  }
}

template <class OutT>
__global__ void sf_features_kernel(SfDev D, int kind, OutT* out) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= D.n) return;
  SfEnv e;
  sf_load_env(D, env, e);
  sf_feature_row(e, D.autoturn != 0, kind, out + (size_t)env * sf_feature_cols(D.autoturn, kind));
}

// out[0, len) <- S[pre, pre + len), by all threads of the block. S is 16-byte aligned and pre = (out / 4) % 4, so out[j] and
// S[pre + j] have the same address mod 16: the 16-byte chunks go out as 16-byte stores, consecutive threads on consecutive
// chunks, and the at most 3 floats at either end as 4-byte stores.
__device__ __forceinline__ void sf_store_span(float* out, const float* S, int pre, int len) {
  const int s1 = pre + len;
  const int v0 = min((pre + 3) & ~3, s1), v1 = max(s1 & ~3, v0);  // [v0, v1): the whole chunks
  for (int s = v0 + 4 * (int)threadIdx.x; s < v1; s += 4 * (int)blockDim.x)
    *reinterpret_cast<float4*>(out + (s - pre)) = *reinterpret_cast<const float4*>(S + s);
  const int k = threadIdx.x;
  if (k < v0 - pre) out[k] = S[pre + k];
  else if (k >= 4 && k - 4 < s1 - v1) out[v1 - pre + k - 4] = S[v1 + k - 4];
}

// ------------------------------------------------------------------------------------------------
// state-only step (render off): one env per thread
// ------------------------------------------------------------------------------------------------
#define SF_STEP_ONLY_BLOCK 128
// The feature rows of step t (the state-only step kernel, all threads of the block): each env's row of its state e.
// In one step the rows of a block's envs are one contiguous span of the output: they are staged in shared memory (two
// buffers, so one barrier per step) and leave as consecutive stores across each warp. One thread storing its own row
// would scatter 4-byte stores 4 * nfeat bytes apart: in HBM, and across PCIe where sf_step_host_features writes straight
// into a page-locked host buffer (~1.7 ns per scattered store, profiles/r02_pcie_write_probe.txt).
__device__ __forceinline__ void sf_feature_rows(const SfDev& D, const SfRollArgs& A, const SfFeatArgs& F, const SfEnv& e, bool mine, int t) {
  __shared__ __align__(16) float rows[2][SF_STEP_ONLY_BLOCK * 19 + 4];  // + 3: the span's offset within 16 bytes
  float* R = rows[t & 1];
  const int b0 = A.env0 + blockIdx.x * SF_STEP_ONLY_BLOCK;
  float* span = F.out + ((size_t)t * D.n + b0) * F.cols;
  const int pre = (int)(((uintptr_t)span >> 2) & 3);
  if (mine) sf_feature_row(e, D.autoturn != 0, F.kind, R + pre + threadIdx.x * F.cols);
  __syncthreads();
  sf_store_span(span, R, pre, min(SF_STEP_ONLY_BLOCK, A.env0 + A.envn - b0) * F.cols);
}

// Agent step t of an env ticks with the one key mask of its action until k ticks have run or one of them ends the
// episode (gym's `frameskip`); index t of the outputs holds the sum of those ticks' rewards and the OR of their done, kill
// and event bits, and FEAT's row t is the state after the agent step. The k iterations are warp-uniform (the loop ends
// early only when no lane of the warp is still ticking), and a lane whose agent step is over just stops ticking: every
// lane reaches the __any_sync of the episode accumulation. The pending Stats increments are 8-bit fields: they are
// flushed every 8 iterations, that is every 8 ticks at most, whatever k is.
// PLAIN (k = 1, no sticky actions, no final observations): the inner loop is one tick and asks no vote. The runtime-k
// loop costs registers: <false, false, false, SF_FINAL_OFF> uses 94 against the plain step's 72, which at 128-thread
// blocks is 20 resident warps per SM instead of 28 on the path that is HBM-bound at T = 1.
// STICKY (sf_set_sticky_actions): before each executed tick the env draws (sf_sticky_hash of its pre-tick rand() count
// and tick); on "stick" the tick runs with the keys the env holds instead of the action's, so it has no press or release
// edges, and the agent step reports SF_EV_STICKY.
// FINAL (sf_set_final_obs, SfFinalMode): IN_KERNEL stores the finished state's agent step index (and feature row) right
// before sf_new_game; DEFERRED (launches of T = 1 only) stores the index, skips the episode accumulation and the new
// game, and marks the env pending: the finished state is stored, drawn by a masked draw launch, and then reset by
// sf_final_reset_kernel exactly as here. Events and shaping do not change: sf_env_step still runs with `autoreset`.
static_assert(SF_CORE_FIRE == SF_KEY_FIRE << 23 && SF_CORE_THRUST == SF_KEY_THRUST << 23 && SF_CORE_LEFT == SF_KEY_LEFT << 23 &&
              SF_CORE_RIGHT == SF_KEY_RIGHT << 23, "the held keys are the key mask at bit 23 of the core word");
template <bool FEAT, bool PLAIN, bool STICKY, int FINAL>
__global__ void __launch_bounds__(SF_STEP_ONLY_BLOCK) sf_step_state_kernel(SfDev D, SfRollArgs A, SfFeatArgs F, int repeat, SfStickyArgs S, SfFinalArgs Z) {
  static_assert(FINAL != SF_FINAL_DEFERRED || !FEAT, "the deferred reset serves the frame route, which has no feature rows");
  static_assert(!PLAIN || (!STICKY && FINAL == SF_FINAL_OFF), "the plain step is one tick of the action's keys");
  const int env = A.env0 + blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool mine = env < A.env0 + A.envn;
  const bool autoreset = !(A.flags & SF_FLAG_NO_AUTORESET), raw = (A.flags & SF_FLAG_RAW_REWARD) != 0;
  const SfHot* H = &D.tab->hot;
  SfEnv e;
  if (mine) sf_load_env(D, env, e);
  int tick = 0;  // iterations run by this warp (the Stats flush cadence)
  for (int t = 0; t < A.T; t++) {
    const int km = mine ? sf_step_keys(D, A, env, t) : 0;
    SfStepOut acc;
    acc.reward = 0; acc.events = 0u; acc.done = false; acc.fort_kill = false;
    bool ticking = mine;
    for (int j = 0; j < (PLAIN ? 1 : repeat) && (PLAIN || __any_sync(0xffffffffu, ticking)); j++, tick++) {
      bool finished = false;
      if (ticking) {
        int keys = km;
        if constexpr (STICKY) {
          if (sf_sticky_hash(S.seed, (unsigned long long)(D.first_global_env + env), (unsigned)e.st3.z, e.q3.z, S.threshold)) {
            keys = ((unsigned)e.q0.x >> 23) & 15;
            acc.events |= SF_EV_STICKY;
          }
        }
        SfStepOut o;
        sf_env_step(D, H, env, e, keys, autoreset, raw, o);
        acc.reward += o.reward; acc.events |= o.events; acc.fort_kill |= o.fort_kill;
        acc.done = o.done; ticking = !o.done;
        finished = o.done && autoreset;
        // the plain step stores its outputs now: kept until after the loop they live across the out-of-line episode
        // accumulation, which made the feature-row instantiation 136 instructions longer and ~2 % slower
        if constexpr (PLAIN) sf_store_step_out(D, A, env, t, o);
      }
      if constexpr (FINAL == SF_FINAL_DEFERRED) {
        if (finished) { Z.step[env] = Z.t0 + t; Z.pending[env] = 1; }
      } else if (__any_sync(0xffffffffu, finished)) {
        sf_accumulate_episode(D, env, e, finished, lane);
        if (finished) {
          if constexpr (FINAL == SF_FINAL_IN_KERNEL) {
            Z.step[env] = Z.t0 + t;
            if constexpr (FEAT) if (Z.rows) sf_feature_row(e, D.autoturn != 0, F.kind, Z.rows + (size_t)env * F.cols);
          }
          sf_new_game(D, H, env, e);
        }
      }
      if (mine && (tick & 7) == 7) sf_flush_stats(D, env, e);
    }
    if (!PLAIN && mine) sf_store_step_out(D, A, env, t, acc);
    if constexpr (FEAT) sf_feature_rows(D, A, F, e, mine, t);
  }
  if (mine) sf_store_env(D, env, e);
}

// The second half of SF_FINAL_DEFERRED's auto-reset, after the finished states have been drawn: the pending envs of
// [env0, env0 + envn) are accumulated and get their new game as in the step kernels (one env per lane; the episode
// statistics are integer sums and a max, so which lanes share a warp reduction does not change them). The step kernel's
// sf_store_env has flushed the pending Stats increments: sf_accumulate_episode reads the counters the in-kernel reset
// reads.
__global__ void __launch_bounds__(SF_STEP_ONLY_BLOCK) sf_final_reset_kernel(SfDev D, unsigned char* pending, int env0, int envn) {
  const int env = env0 + blockIdx.x * blockDim.x + threadIdx.x;
  const bool finished = env < env0 + envn && pending[env];
  if (!__any_sync(0xffffffffu, finished)) return;
  SfEnv e;
  if (finished) sf_load_env(D, env, e);
  sf_accumulate_episode(D, env, e, finished, threadIdx.x & 31);
  if (finished) {
    sf_new_game(D, &D.tab->hot, env, e);
    sf_store_env(D, env, e);
    pending[env] = 0;
  }
}

// ---- state records (AoS <-> SoA), one thread per env ----
__global__ void sf_get_state_kernel(SfDev D, int first, int count, sf_state_record* out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const int i = first + k;
  const SfTables* T = D.tab;
  SfEnv e;
  sf_load_env(D, i, e);
  sf_state_record r;
  memset(&r, 0, sizeof(r));
  unsigned core = (unsigned)e.q0.x;
  r.ship_x = e.pos.x; r.ship_y = e.pos.y; r.ship_vx = e.vel.x; r.ship_vy = e.vel.y;
  r.ship_angle = (double)(core & SF_CORE_ANGLE_MASK);
  r.fortress_angle = 10.0 * ((core >> SF_CORE_FANG_SHIFT) & 63u);
  r.fortress_last_angle = 10.0 * ((core >> SF_CORE_FLAST_SHIFT) & 63u);
  r.missile_mask = (unsigned)e.q0.y & SF_PMASK_MISSILES;
  r.shell_mask = ((unsigned)e.q0.y >> SF_PMASK_SHELL_SHIFT) & 0xFu;
  for (int s = 0; s < SF_MAX_MISSILES; s++) if ((r.missile_mask >> s) & 1) {
    double2 p = D.mpos[(size_t)s * D.n_pad + i];
    int a = D.mang[(size_t)s * D.n_pad + i];
    r.missile_x[s] = p.x; r.missile_y[s] = p.y; r.missile_angle[s] = a;
    r.missile_vx[s] = SF_DMUL(20.0, T->cos_deg[a]); r.missile_vy[s] = SF_DMUL(20.0, T->sin_deg[a]);
  }
  for (int s = 0; s < SF_DEV_SHELLS; s++) if ((r.shell_mask >> s) & 1) {
    double2 p = D.spos[(size_t)s * D.n_pad + i], v = D.svel[(size_t)s * D.n_pad + i];
    r.shell_x[s] = p.x; r.shell_y[s] = p.y; r.shell_vx[s] = v.x; r.shell_vy[s] = v.y;
    r.shell_angle[s] = D.sang[(size_t)s * D.n_pad + i];
  }
  r.points = __int_as_float(e.q3.x); r.raw_points = __int_as_float(e.q3.y);
  r.ship_alive = (core & SF_CORE_SHIP_ALIVE) != 0; r.fortress_alive = (core & SF_CORE_FORT_ALIVE) != 0;
  r.ship_death_timer = e.q0.z;
  r.fire_timer = e.q2.x; r.thrust_timer = e.q2.y; r.left_timer = e.q2.z; r.right_timer = e.q2.w;
  r.thrust_flag = (core & SF_CORE_THRUST) != 0; r.fire_flag = (core & SF_CORE_FIRE) != 0;
  r.left_flag = (core & SF_CORE_LEFT) != 0; r.right_flag = (core & SF_CORE_RIGHT) != 0;
  r.turn_flag = (r.left_flag && !r.right_flag) ? 1 : (!r.left_flag && r.right_flag) ? 2 : 0;  // game.cpp:265-270
  r.fortress_timer = e.q0.w; r.fortress_death_timer = e.q1.x; r.fortress_vuln_timer = e.q1.y;
  r.vulnerability = e.q1.z; r.tick = e.q3.z; r.time = e.q3.z * SF_TICK_MS;
  const int4 st0 = D.st0[i], st1 = D.st1[i], st2 = D.st2[i];
  r.stats[0] = st0.x; r.stats[1] = st0.y; r.stats[2] = st0.z; r.stats[3] = st0.w;
  r.stats[4] = st1.x; r.stats[5] = st1.y; r.stats[6] = st1.z; r.stats[7] = st1.w;
  r.stats[8] = st2.x; r.stats[9] = st2.y; r.stats[10] = st2.z; r.stats[11] = st2.w;
  r.stats[12] = e.st3.x;
  r.prev_vlner = e.q1.w;
  r.rng_seed = (unsigned)e.st3.w; r.rng_count = (unsigned)e.st3.z;
  r.ep_return = e.q3.w;
  out[k] = r;
}

__global__ void sf_set_state_kernel(SfDev D, int first, int count, const sf_state_record* in) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const int i = first + k;
  const sf_state_record& r = in[k];
  SfEnv e;
  sf_load_env(D, i, e);
  // the rand stream is re-derived from (seed, count)
  if ((unsigned)e.st3.w != r.rng_seed || (unsigned)e.st3.z > r.rng_count) sf_srand(D, i, e, r.rng_seed);
  while ((unsigned)e.st3.z < r.rng_count) (void)sf_rand(D, i, e);
  unsigned core = ((unsigned)(int)r.ship_angle & SF_CORE_ANGLE_MASK) | (((unsigned)(int)(r.fortress_angle / 10.0) & 63u) << SF_CORE_FANG_SHIFT) |
                  (((unsigned)(int)(r.fortress_last_angle / 10.0) & 63u) << SF_CORE_FLAST_SHIFT);
  if (r.ship_alive) core |= SF_CORE_SHIP_ALIVE;
  if (r.fortress_alive) core |= SF_CORE_FORT_ALIVE;
  if (r.fire_flag) core |= SF_CORE_FIRE;
  if (r.thrust_flag) core |= SF_CORE_THRUST;
  if (r.left_flag) core |= SF_CORE_LEFT;
  if (r.right_flag) core |= SF_CORE_RIGHT;
  e.pos = make_double2(r.ship_x, r.ship_y); e.vel = make_double2(r.ship_vx, r.ship_vy);
  e.q0 = make_int4((int)core, (int)((r.missile_mask & SF_PMASK_MISSILES) | ((r.shell_mask & 0xFu) << SF_PMASK_SHELL_SHIFT)), r.ship_death_timer, r.fortress_timer);
  e.q1 = make_int4(r.fortress_death_timer, r.fortress_vuln_timer, r.vulnerability, r.prev_vlner);
  e.q2 = make_int4(r.fire_timer, r.thrust_timer, r.left_timer, r.right_timer);
  e.q3 = make_int4(__float_as_int(r.points), __float_as_int(r.raw_points), r.tick, r.ep_return);
  D.st0[i] = make_int4(r.stats[0], r.stats[1], r.stats[2], r.stats[3]);
  D.st1[i] = make_int4(r.stats[4], r.stats[5], r.stats[6], r.stats[7]);
  D.st2[i] = make_int4(r.stats[8], r.stats[9], r.stats[10], r.stats[11]);
  e.st3.x = r.stats[12];
  for (int s = 0; s < SF_MAX_MISSILES; s++) if ((r.missile_mask >> s) & 1) {
    D.mpos[(size_t)s * D.n_pad + i] = make_double2(r.missile_x[s], r.missile_y[s]);
    D.mang[(size_t)s * D.n_pad + i] = (short)(int)r.missile_angle[s];
  }
  for (int s = 0; s < SF_DEV_SHELLS; s++) if ((r.shell_mask >> s) & 1) {
    D.spos[(size_t)s * D.n_pad + i] = make_double2(r.shell_x[s], r.shell_y[s]);
    D.svel[(size_t)s * D.n_pad + i] = make_double2(r.shell_vx[s], r.shell_vy[s]);
    D.sang[(size_t)s * D.n_pad + i] = r.shell_angle[s];
  }
  sf_forget_render_caches(D, i);
  sf_store_env(D, i, e);
}

// ---- env blobs (sf_save_envs / sf_load_envs): SoA <-> one SF_ENV_BLOB_BYTES row per env, layout in sf_b200.h ----
// One warp per block moves a tile of 32 envs through shared memory. On the SoA side lane l handles env l of the tile (a
// warp access is 512 B per int4 array and 128 B per rand() word when the indices are contiguous); on the blob side the
// lanes run over the 16-byte chunks of the tile's 32 consecutive rows, so the rows are read and written fully coalesced.
// Global -> shared moves are cp.async: a warp has the whole tile in flight without holding it in registers.
#define SF_BLOB_CHUNKS (SF_ENV_BLOB_BYTES / 16)
#define SF_BLOB_PITCH (SF_BLOB_CHUNKS + 1)  // shared row pitch in chunks: odd, so the 8 lanes of a 16-byte phase hit 8 bank quads
#define SF_BLOB_BLOCKS_PER_SM 8             // 8 x 27 KB of shared memory
enum { SF_BO_POS = 16, SF_BO_VEL = 32, SF_BO_Q = 48, SF_BO_ST = 112, SF_BO_MPOS = 176, SF_BO_SPOS = 496, SF_BO_SVEL = 560,
       SF_BO_SANG = 624, SF_BO_MANG = 656, SF_BO_RNG = 696, SF_BO_END = 820 };
static_assert(SF_BO_MANG + 2 * SF_MAX_MISSILES == SF_BO_RNG && SF_BO_RNG + 4 * SF_RNG_WORDS == SF_BO_END, "blob layout");
static_assert(SF_BO_END <= SF_ENV_BLOB_BYTES && SF_ENV_BLOB_BYTES % 16 == 0, "blob size");

__device__ __forceinline__ void sf_cp_async(void* smem, const void* gmem, int bytes) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  if (bytes == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
  else if (bytes == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void sf_cp_async_wait() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

__global__ void __launch_bounds__(32) sf_save_envs_kernel(SfDev D, int gametype, const int* __restrict__ idx, int count, int4* __restrict__ blob) {
  __shared__ int4 tile[32 * SF_BLOB_PITCH];
  const int lane = threadIdx.x;
  const size_t np = (size_t)D.n_pad;
  int4* row = tile + lane * SF_BLOB_PITCH;
  char* rb = reinterpret_cast<char*>(row);
  const int4 z = make_int4(0, 0, 0, 0);
  for (int base = blockIdx.x * 32; base < count; base += gridDim.x * 32) {
    const int k = base + lane;
    const int i = k < count ? (idx ? idx[k] : k) : -1;
    if (i >= 0 && i < D.n) {
      const int4 q0 = D.q0[i];
      const unsigned pm = (unsigned)q0.y;
      row[0] = make_int4((int)SF_ENV_BLOB_MAGIC, SF_ENV_BLOB_VERSION, gametype, 0);
      sf_cp_async(rb + SF_BO_POS, &D.pos[i], 16);
      sf_cp_async(rb + SF_BO_VEL, &D.vel[i], 16);
      row[SF_BO_Q / 16] = q0;
      sf_cp_async(rb + SF_BO_Q + 16, &D.q1[i], 16);
      sf_cp_async(rb + SF_BO_Q + 32, &D.q2[i], 16);
      sf_cp_async(rb + SF_BO_Q + 48, &D.q3[i], 16);
      sf_cp_async(rb + SF_BO_ST, &D.st0[i], 16);
      sf_cp_async(rb + SF_BO_ST + 16, &D.st1[i], 16);
      sf_cp_async(rb + SF_BO_ST + 32, &D.st2[i], 16);
      sf_cp_async(rb + SF_BO_ST + 48, &D.st3[i], 16);
      short* mang = reinterpret_cast<short*>(rb + SF_BO_MANG);
#pragma unroll
      for (int s = 0; s < SF_MAX_MISSILES; s++) {
        const bool live = (pm >> s) & 1u;
        if (live) sf_cp_async(rb + SF_BO_MPOS + 16 * s, &D.mpos[s * np + i], 16);
        else row[SF_BO_MPOS / 16 + s] = z;  // dead slots are zero: equal states give equal rows
        mang[s] = live ? D.mang[s * np + i] : (short)0;
      }
#pragma unroll
      for (int s = 0; s < SF_DEV_SHELLS; s++) {
        if ((pm >> (SF_PMASK_SHELL_SHIFT + s)) & 1u) {
          sf_cp_async(rb + SF_BO_SPOS + 16 * s, &D.spos[s * np + i], 16);
          sf_cp_async(rb + SF_BO_SVEL + 16 * s, &D.svel[s * np + i], 16);
          sf_cp_async(rb + SF_BO_SANG + 8 * s, &D.sang[s * np + i], 8);
        } else {
          row[SF_BO_SPOS / 16 + s] = z;
          row[SF_BO_SVEL / 16 + s] = z;
          reinterpret_cast<double*>(rb + SF_BO_SANG)[s] = 0.0;
        }
      }
#pragma unroll
      for (int w = 0; w < SF_RNG_WORDS; w++) sf_cp_async(rb + SF_BO_RNG + 4 * w, &D.rng[w * np + i], 4);
      for (int b = SF_BO_END; b < SF_ENV_BLOB_BYTES; b += 4) *reinterpret_cast<int*>(rb + b) = 0;
    } else if (k < count) {
      for (int c = 0; c < SF_BLOB_CHUNKS; c++) row[c] = z;  // no such env
    }
    sf_cp_async_wait();
    __syncwarp();
    const int rows = min(32, count - base);
    int4* out = blob + (size_t)base * SF_BLOB_CHUNKS;
#pragma unroll 4
    for (int c = lane; c < rows * SF_BLOB_CHUNKS; c += 32) {
      const int r = c / SF_BLOB_CHUNKS;
      out[c] = tile[r * SF_BLOB_PITCH + (c - r * SF_BLOB_CHUNKS)];
    }
    __syncwarp();  // the tile is reused
  }
}

// Rows with a bad header or target index are skipped and counted into *rejected (one atomic per warp). Writes only the
// live missile and shell slots (the others are never read), and resets the env's render caches.
__global__ void __launch_bounds__(32) sf_load_envs_kernel(SfDev D, int gametype, const int4* __restrict__ blob, const int* __restrict__ idx, int count,
                                                          int* rejected) {
  __shared__ int4 tile[32 * SF_BLOB_PITCH];
  const int lane = threadIdx.x;
  const size_t np = (size_t)D.n_pad;
  const int4* row = tile + lane * SF_BLOB_PITCH;
  const char* rb = reinterpret_cast<const char*>(row);
  for (int base = blockIdx.x * 32; base < count; base += gridDim.x * 32) {
    const int rows = min(32, count - base);
    const int4* in = blob + (size_t)base * SF_BLOB_CHUNKS;
#pragma unroll 4
    for (int c = lane; c < rows * SF_BLOB_CHUNKS; c += 32) {
      const int r = c / SF_BLOB_CHUNKS;
      sf_cp_async(&tile[r * SF_BLOB_PITCH + (c - r * SF_BLOB_CHUNKS)], &in[c], 16);
    }
    sf_cp_async_wait();
    __syncwarp();
    const int k = base + lane;
    const int i = k < count ? (idx ? idx[k] : k) : -1;
    bool ok = false;
    if (k < count) {
      const int4 hd = row[0];
      ok = (unsigned)hd.x == SF_ENV_BLOB_MAGIC && hd.y == SF_ENV_BLOB_VERSION && hd.z == gametype && i >= 0 && i < D.n;
    }
    const unsigned bad = __ballot_sync(0xFFFFFFFFu, k < count && !ok);
    if (lane == 0 && bad && rejected) atomicAdd(rejected, __popc(bad));
    if (ok) {
      const int4 q0 = row[SF_BO_Q / 16];
      const unsigned pm = (unsigned)q0.y;
      D.pos[i] = *reinterpret_cast<const double2*>(rb + SF_BO_POS);
      D.vel[i] = *reinterpret_cast<const double2*>(rb + SF_BO_VEL);
      D.q0[i] = q0;
      D.q1[i] = row[SF_BO_Q / 16 + 1];
      D.q2[i] = row[SF_BO_Q / 16 + 2];
      D.q3[i] = row[SF_BO_Q / 16 + 3];
      D.st0[i] = row[SF_BO_ST / 16];
      D.st1[i] = row[SF_BO_ST / 16 + 1];
      D.st2[i] = row[SF_BO_ST / 16 + 2];
      D.st3[i] = row[SF_BO_ST / 16 + 3];
      const short* mang = reinterpret_cast<const short*>(rb + SF_BO_MANG);
#pragma unroll
      for (int s = 0; s < SF_MAX_MISSILES; s++) if ((pm >> s) & 1u) {
        D.mpos[s * np + i] = *reinterpret_cast<const double2*>(rb + SF_BO_MPOS + 16 * s);
        D.mang[s * np + i] = mang[s];
      }
#pragma unroll
      for (int s = 0; s < SF_DEV_SHELLS; s++) if ((pm >> (SF_PMASK_SHELL_SHIFT + s)) & 1u) {
        D.spos[s * np + i] = *reinterpret_cast<const double2*>(rb + SF_BO_SPOS + 16 * s);
        D.svel[s * np + i] = *reinterpret_cast<const double2*>(rb + SF_BO_SVEL + 16 * s);
        D.sang[s * np + i] = reinterpret_cast<const double*>(rb + SF_BO_SANG)[s];
      }
      const unsigned* rng = reinterpret_cast<const unsigned*>(rb + SF_BO_RNG);
#pragma unroll
      for (int w = 0; w < SF_RNG_WORDS; w++) D.rng[w * np + i] = rng[w];
      sf_forget_render_caches(D, i);
    }
    __syncwarp();  // the tile is reused
  }
}

// ================================================================================================
// C-ABI
// ================================================================================================
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CUDA_TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(SF_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

#define SF_MAX_MIRRORS 4
#define SF_HOST_STEP_SLICES 4  // sf_step_host with whole frames: launches over slices of the slab (see there)
struct sf_handle {
  SfDev dev;
  int device;
  int action_set;
  int gametype;  // 0 youturn 1 autoturn 2 test-youturn 3 test-autoturn
  int num_sms;
  int action_repeat;  // ticks per agent step of every stepping entry point (sf_set_action_repeat), 1 by default
  double sticky_p;      // sf_set_sticky_actions: p, and the kernel's form of (p, seed); 0 by default
  SfStickyArgs sticky;
  // sf_set_final_obs: the caller's device buffers (step == NULL: off), and the deferred reset's marks (uint8[n], zero
  // between calls)
  struct FinalObs { uint8_t* frames; float* rows; int32_t* step; } final_obs;
  unsigned char* d_final_pending;
  void* slab;
  size_t slab_bytes;
  SfTables* h_tab;
  // pinned staging for sf_step_host
  int* d_actions; unsigned char* d_obs; int* d_reward; unsigned char* d_done; unsigned char* d_kill; unsigned* d_events;
  size_t staging_obs_bytes;
  SfSched* d_sched;  // sf_rollout_kernel's scheduling state (group hand-out, cost-dealt envs)
  cudaStream_t host_compute, host_copy;  // sf_step_host: kernels of slice k + 1 overlap the device->host copy of slice k
  cudaEvent_t host_ev[SF_HOST_STEP_SLICES];
  // SF_FLAG_HOST_DELTA: device copy of what the caller's page-locked h_obs holds, so that only changed bytes cross PCIe
  struct Mirror { const void* host; unsigned char* d; size_t cap, bytes; unsigned long long used; };  // host: the buffer it describes, or NULL
  Mirror mirrors[SF_MAX_MIRRORS];     // one per host buffer (a caller may rotate a few buffers); least recently used goes first
  unsigned long long mirror_clock;
  unsigned long long* d_delta_stats;  // [0] observation bytes written to the host by delta calls, [1] delta calls
  unsigned long long full_calls;      // calls that sent whole frames (first call, new buffer, flag absent)

  // The mirror of host buffer `host`, with room for `bytes`: its own entry, else a free one, else the least recently used
  // one. An entry that is taken over or grown describes no buffer until whole frames have been copied into it.
  int mirror_for(const void* host, size_t bytes, Mirror** out) {
    Mirror* mir = nullptr;
    for (auto& m : mirrors) if (m.host == host) mir = &m;
    if (!mir) {
      for (auto& m : mirrors) if (!mir || (mir->host && (!m.host || m.used < mir->used))) mir = &m;
      mir->host = nullptr;
    }
    if (bytes > mir->cap) {
      if (mir->d) { cudaFree(mir->d); mir->d = nullptr; mir->cap = 0; }
      mir->host = nullptr;
      CUDA_TRY(cudaMalloc(&mir->d, bytes));
      mir->cap = bytes;
    }
    mir->used = ++mirror_clock;
    *out = mir;
    return SF_OK;
  }
  void forget_mirrors(const void* host) {  // NULL: every buffer; the device memory is kept for the next buffer
    for (auto& m : mirrors) if (m.host == host || !host) m.host = nullptr;
  }
};

extern "C" const char* sf_last_error(void) { return g_err.c_str(); }
extern "C" int sf_version(void) { return 100; }

static int gametype_of(const char* s) {
  if (!s) return -1;
  if (!strcmp(s, "youturn")) return 0;
  if (!strcmp(s, "autoturn")) return 1;
  if (!strcmp(s, "test-youturn")) return 2;
  if (!strcmp(s, "test-autoturn")) return 3;
  return -1;
}

// P2: action tables (ssf_env.py:65-90)
static int build_actions(int gametype, int action_set, int* km) {
  bool youturn = gametype == 0 || gametype == 2;
  if (action_set == 1) {
    const int tab[5] = {0, SF_KEY_FIRE, SF_KEY_THRUST, SF_KEY_LEFT, SF_KEY_RIGHT};
    int n = youturn ? 5 : 3;
    for (int i = 0; i < n; i++) km[i] = tab[i];
    return n;
  }
  if (action_set == 0 && !youturn) {  // np.meshgrid([0,1],[0,1]).T.reshape(-1,2): fire = bit 1, thrust = bit 0
    for (int a = 0; a < 4; a++) km[a] = ((a >> 1) & 1 ? SF_KEY_FIRE : 0) | ((a & 1) ? SF_KEY_THRUST : 0);
    return 4;
  }
  if (action_set == 0 || action_set == -1) {  // 4-key meshgrid: row = right*8 + left*4 + fire*2 + thrust
    for (int a = 0; a < 16; a++) {
      int m = ((a >> 1) & 1 ? SF_KEY_FIRE : 0) | ((a & 1) ? SF_KEY_THRUST : 0) | ((a >> 2) & 1 ? SF_KEY_LEFT : 0) | ((a >> 3) & 1 ? SF_KEY_RIGHT : 0);
      km[a] = youturn ? m : (m & (SF_KEY_FIRE | SF_KEY_THRUST));
    }
    return 16;
  }
  return -1;
}

template <class T>
static T* carve(char*& p, size_t count) {
  T* r = reinterpret_cast<T*>(p);
  size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
  p += bytes;
  return r;
}

static size_t layout(SfDev& d, char* base) {
  char* p = base;
  size_t np = (size_t)d.n_pad;
  d.pos = carve<double2>(p, np); d.vel = carve<double2>(p, np);
  d.q0 = carve<int4>(p, np); d.q1 = carve<int4>(p, np); d.q2 = carve<int4>(p, np); d.q3 = carve<int4>(p, np);
  d.st0 = carve<int4>(p, np); d.st1 = carve<int4>(p, np); d.st2 = carve<int4>(p, np); d.st3 = carve<int4>(p, np);
  d.mpos = carve<double2>(p, np * SF_MAX_MISSILES); d.mang = carve<short>(p, np * SF_MAX_MISSILES);
  d.spos = carve<double2>(p, np * SF_DEV_SHELLS); d.svel = carve<double2>(p, np * SF_DEV_SHELLS); d.sang = carve<double>(p, np * SF_DEV_SHELLS);
  d.rng = carve<unsigned>(p, np * SF_RNG_WORDS);
  d.expc = carve<unsigned char>(p, np * SF_EXP_W * SF_EXP_W);
  d.expstamp = carve<unsigned>(p, np);
  d.expo = carve<unsigned char>(p, np * SF_EXPO_BYTES);
  d.expo_meta = carve<uint2>(p, np);
  d.epi = carve<unsigned long long>(p, SF_NUM_EPISODE_STATS);
  d.tab = carve<SfTables>(p, 1);
  d.static_image = carve<unsigned char>(p, SF_STATIC_BYTES);
  return (size_t)(p - base);
}

extern "C" int sf_destroy(sf_handle* h);

extern "C" int sf_create(const char* gametype, int action_set, int n_envs, int device, sf_handle** out) {
  if (!out) return fail(SF_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int gt = gametype_of(gametype);
  if (gt < 0) return fail(SF_ERR_INVALID, std::string("cannot initialize Game. Unknown config value: `") + (gametype ? gametype : "(null)") + "'");
  if (n_envs <= 0) return fail(SF_ERR_INVALID, "n_envs must be positive");
  int km[16];
  int na = build_actions(gt, action_set, km);
  if (na < 0) return fail(SF_ERR_INVALID, "action_set must be 1, 0 or -1");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(SF_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)");
  CUDA_TRY(cudaSetDevice(device));
  int num_sms = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));

  sf_handle* h = new sf_handle();
  memset(h, 0, sizeof(*h));
  h->device = device; h->num_sms = num_sms > 0 ? num_sms : 148; h->action_set = action_set; h->gametype = gt;
  h->action_repeat = 1;
  SfDev& d = h->dev;
  d.n = n_envs; d.n_pad = (n_envs + 31) & ~31;
  d.autoturn = (gt == 1 || gt == 3);
  bool test = gt >= 2;
  d.shaped = !test;                      // ssf_env.py:235
  d.destroy_fortress = test ? 100 : 1;   // configs.cpp:8,57,68
  d.death_penalty = test ? 100 : 1;      // configs.cpp:9,58,69
  d.missile_penalty = test ? 2.0f : (float)0.05;  // configs.cpp:10,59,70 (double -> float parameter, game.cpp:104)
  d.num_actions = na;
  for (int i = 0; i < 16; i++) d.keymask_of_action[i] = i < na ? km[i] : 0;
  d.first_global_env = 0;

  h->h_tab = new SfTables();
  char err[256] = {0};
  if (sf_build_tables(h->h_tab, err, sizeof(err))) { std::string m = err; delete h->h_tab; delete h; return fail(SF_ERR_INVALID, "table build failed: " + m); }

  // every failure below releases what has been allocated (sf_destroy frees whatever is non-NULL)
  auto bail = [&](const char* what, cudaError_t ce) { std::string m = std::string(what) + ": " + cudaGetErrorString(ce); sf_destroy(h); return fail(SF_ERR_CUDA, m); };
  cudaError_t ce;
  h->slab_bytes = layout(d, nullptr);
  if ((ce = cudaMalloc(&h->slab, h->slab_bytes)) != cudaSuccess) return bail("cudaMalloc state slab", ce);
  layout(d, (char*)h->slab);
  if ((ce = cudaMalloc(&h->d_sched, sizeof(SfSched))) != cudaSuccess) return bail("cudaMalloc scheduler state", ce);
  if ((ce = cudaMemset(h->d_sched, 0, sizeof(SfSched))) != cudaSuccess) return bail("cudaMemset scheduler state", ce);
  if ((ce = cudaMemset(h->slab, 0, h->slab_bytes)) != cudaSuccess) return bail("cudaMemset state slab", ce);
  if ((ce = cudaMemcpy((void*)d.tab, h->h_tab, sizeof(SfTables), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("upload tables", ce);
  if ((ce = cudaFuncSetAttribute(sf_rollout_kernel<SF_ROLL_STEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS))) != cudaSuccess) return bail("shared memory opt-in (rollout)", ce);
  if ((ce = cudaFuncSetAttribute(sf_rollout_kernel<SF_ROLL_STEP_HOST_DELTA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS))) != cudaSuccess) return bail("shared memory opt-in (rollout, host delta)", ce);
  if ((ce = cudaFuncSetAttribute(sf_rollout_kernel<SF_ROLL_DRAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS))) != cudaSuccess) return bail("shared memory opt-in (rollout, draw)", ce);
  if ((ce = cudaFuncSetAttribute(sf_pack_static_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS))) != cudaSuccess) return bail("shared memory opt-in (pack)", ce);
  if ((ce = cudaFuncSetAttribute(sf_save_envs_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared)) != cudaSuccess) return bail("shared memory carveout (save envs)", ce);
  if ((ce = cudaFuncSetAttribute(sf_load_envs_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared)) != cudaSuccess) return bail("shared memory carveout (load envs)", ce);
  sf_pack_static_kernel<<<1, SF_BLOCK, SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS)>>>(d, const_cast<unsigned char*>(d.static_image));
  if ((ce = cudaGetLastError()) != cudaSuccess) return bail("static image kernel launch", ce);
  // default seeding: every env replays srand(1) — the reference never seeds libc (game.cpp:137-148)
  sf_seed_kernel<<<(d.n + 127) / 128, 128>>>(d, nullptr);
  if ((ce = cudaGetLastError()) != cudaSuccess) return bail("seed kernel launch", ce);
  if ((ce = cudaDeviceSynchronize()) != cudaSuccess) return bail("seed kernel", ce);
  *out = h;
  return SF_OK;
}

extern "C" int sf_destroy(sf_handle* h) {
  if (!h) return SF_OK;
  cudaSetDevice(h->device);
  if (h->slab) cudaFree(h->slab);
  if (h->d_actions) cudaFree(h->d_actions);
  if (h->d_obs) cudaFree(h->d_obs);
  if (h->d_reward) cudaFree(h->d_reward);
  if (h->d_done) cudaFree(h->d_done);
  if (h->d_kill) cudaFree(h->d_kill);
  if (h->d_events) cudaFree(h->d_events);
  if (h->d_sched) cudaFree(h->d_sched);
  if (h->d_final_pending) cudaFree(h->d_final_pending);
  for (auto& m : h->mirrors) if (m.d) cudaFree(m.d);
  if (h->d_delta_stats) cudaFree(h->d_delta_stats);
  if (h->host_compute) cudaStreamDestroy(h->host_compute);
  if (h->host_copy) cudaStreamDestroy(h->host_copy);
  for (int k = 0; k < SF_HOST_STEP_SLICES; k++) if (h->host_ev[k]) cudaEventDestroy(h->host_ev[k]);
  delete h->h_tab;
  delete h;
  return SF_OK;
}

extern "C" int sf_num_envs(const sf_handle* h) { return h ? h->dev.n : -1; }
extern "C" int sf_num_actions(const sf_handle* h) { return h ? h->dev.num_actions : -1; }
extern "C" int sf_action_keymask(const sf_handle* h, int action) {
  if (!h || action < 0 || action >= h->dev.num_actions) return -1;
  return h->dev.keymask_of_action[action];
}
extern "C" long long sf_state_bytes(const sf_handle* h) { return h ? (long long)h->slab_bytes : -1; }

extern "C" int sf_seed(sf_handle* h, const uint32_t* h_seeds, long long first_global_env, void* stream) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  h->dev.first_global_env = first_global_env;
  unsigned* d_seeds = nullptr;
  cudaError_t ce = cudaSuccess;
  if (h_seeds) {
    CUDA_TRY(cudaMalloc(&d_seeds, sizeof(unsigned) * h->dev.n));
    ce = cudaMemcpyAsync(d_seeds, h_seeds, sizeof(unsigned) * h->dev.n, cudaMemcpyHostToDevice, st);
  }
  if (ce == cudaSuccess) {
    sf_seed_kernel<<<(h->dev.n + 127) / 128, 128, 0, st>>>(h->dev, d_seeds);
    ce = cudaGetLastError();
  }
  if (d_seeds) {  // the temporary is released on every path
    cudaError_t cs = cudaStreamSynchronize(st);
    if (ce == cudaSuccess) ce = cs;
    cudaFree(d_seeds);
  }
  if (ce != cudaSuccess) return fail(SF_ERR_CUDA, std::string("sf_seed: ") + cudaGetErrorString(ce));
  return SF_OK;
}

// Envs per group (= per block and tick). While every group can have its own SM the envs are spread evenly over
// the SMs (4096 envs -> 28 per block, 147 blocks); beyond that a group is a full warp of 32 stepping lanes and
// the blocks are persistent over their groups.
static void group_shape(const sf_handle* h, int n, int* EB, int* ngroups, int* blocks) {
  const int sms = h->num_sms;  // one block per SM
  const int eb = n <= sms * SF_GROUP_ENVS ? (n + sms - 1) / sms : SF_GROUP_ENVS;
  *EB = eb;
  *ngroups = (n + eb - 1) / eb;
  *blocks = std::min(*ngroups, sms);
}

// Whether frames come from separate launches: the state kernel for each agent step, then a SF_ROLL_DRAW of the state it
// left (action repeat k > 1, sticky actions with p > 0, or final observations), rather than from the fused kernel. The
// fused kernel's stepping warp is its critical side already: k ticks per drawn tick would make it the bottleneck
// (DESIGN.md 4.6). (A p below 2^-33 rounds to threshold 0, which never sticks: the fused kernel gives the same bits.)
static bool frames_need_split(const sf_handle* h) {
  return h->action_repeat > 1 || h->sticky.threshold > 0 || h->final_obs.step;
}

// The state-only step of a.T agent steps. step0: the call's agent step index of a's step 0 (final_step's values).
static int launch_state(sf_handle* h, const SfRollArgs& a, const SfFeatArgs& f, int final_mode, int step0, cudaStream_t st) {
  typedef void (*Kernel)(SfDev, SfRollArgs, SfFeatArgs, int, SfStickyArgs, SfFinalArgs);
  // [FEAT][STICKY][final mode]; the deferred reset serves the frame route, which has no feature rows
  static const Kernel kernels[2][2][3] = {
      {{sf_step_state_kernel<false, false, false, SF_FINAL_OFF>, sf_step_state_kernel<false, false, false, SF_FINAL_IN_KERNEL>,
        sf_step_state_kernel<false, false, false, SF_FINAL_DEFERRED>},
       {sf_step_state_kernel<false, false, true, SF_FINAL_OFF>, sf_step_state_kernel<false, false, true, SF_FINAL_IN_KERNEL>,
        sf_step_state_kernel<false, false, true, SF_FINAL_DEFERRED>}},
      {{sf_step_state_kernel<true, false, false, SF_FINAL_OFF>, sf_step_state_kernel<true, false, false, SF_FINAL_IN_KERNEL>, nullptr},
       {sf_step_state_kernel<true, false, true, SF_FINAL_OFF>, sf_step_state_kernel<true, false, true, SF_FINAL_IN_KERNEL>, nullptr}}};
  static const Kernel plain_kernels[2] = {sf_step_state_kernel<false, true, false, SF_FINAL_OFF>, sf_step_state_kernel<true, true, false, SF_FINAL_OFF>};
  const bool feat = f.out != nullptr, sticky = h->sticky.threshold > 0;
  const bool plain = h->action_repeat == 1 && !sticky && final_mode == SF_FINAL_OFF;
  const Kernel k = plain ? plain_kernels[feat] : kernels[feat][sticky][final_mode];
  const sf_handle::FinalObs& fo = h->final_obs;
  const SfFinalArgs z = {fo.step, feat ? fo.rows : nullptr, h->d_final_pending, step0};
  k<<<(a.envn + SF_STEP_ONLY_BLOCK - 1) / SF_STEP_ONLY_BLOCK, SF_STEP_ONLY_BLOCK, 0, st>>>(h->dev, a, f, h->action_repeat, h->sticky, z);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

// SF_ROLL_DRAW: the frames of the current state (a.T = 1) of the envs a.draw_mask selects (NULL: all), static groups
static int launch_draw(sf_handle* h, SfRollArgs a, cudaStream_t st) {
  int blocks;
  group_shape(h, a.envn, &a.EB, &a.ngroups, &blocks);
  a.sched = nullptr;
  sf_rollout_kernel<SF_ROLL_DRAW><<<blocks, SF_BLOCK, SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS), st>>>(h->dev, a);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

// The fused step + render of a.T agent steps of one tick. The hand-out counters serve full-slab steps only; slices of the
// slab (sf_step_host) and in-kernel delta launches take static groups.
static int launch_fused(sf_handle* h, SfRollArgs a, cudaStream_t st) {
  int blocks;
  group_shape(h, a.envn, &a.EB, &a.ngroups, &blocks);
  a.sched = (a.env0 == 0 && a.envn == h->dev.n && !a.host_obs) ? h->d_sched : nullptr;
  if (a.host_obs) sf_rollout_kernel<SF_ROLL_STEP_HOST_DELTA><<<blocks, SF_BLOCK, SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS), st>>>(h->dev, a);
  else sf_rollout_kernel<SF_ROLL_STEP><<<blocks, SF_BLOCK, SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS), st>>>(h->dev, a);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

// a.T agent steps of [a.env0, a.env0 + a.envn): the launches of every stepping entry point. Frames when a.flags has
// SF_FLAG_RENDER and a.obs is set; f: feature rows (render off only). Only enqueues on st (CUDA graph capture).
static int launch_steps(sf_handle* h, const SfRollArgs& a, const SfFeatArgs& f, cudaStream_t st) {
  const sf_handle::FinalObs& fo = h->final_obs;
  const bool render = (a.flags & SF_FLAG_RENDER) && a.obs, autoreset = !(a.flags & SF_FLAG_NO_AUTORESET);
  if (fo.step) {  // one end per env and call at most, so one slot per env is exact (sf_set_final_obs)
    if ((long long)a.T * h->action_repeat > SF_GAME_TICKS)
      return fail(SF_ERR_INVALID, "final observations: T * action_repeat must be <= " + std::to_string(SF_GAME_TICKS) + " (one episode end per env and call)");
    CUDA_TRY(cudaMemsetAsync(fo.step + a.env0, 0xFF, sizeof(int32_t) * (size_t)a.envn, st));
  }
  // With final frames the state kernel defers the auto-reset: a masked draw of the finished states and
  // sf_final_reset_kernel come between it and the step's draw (DESIGN.md 4.8).
  const bool deferred = fo.step && render && fo.frames && autoreset;
  const int final_mode = (!fo.step || !autoreset) ? SF_FINAL_OFF : deferred ? SF_FINAL_DEFERRED : SF_FINAL_IN_KERNEL;
  if (!render) return launch_state(h, a, f, final_mode, 0, st);
  if (!frames_need_split(h)) return launch_fused(h, a, st);
  const size_t n = (size_t)h->dev.n, per = (a.flags & SF_FLAG_NATIVE_OBS) ? (size_t)SF_NAT_H * SF_NAT_W : (size_t)84 * 84;
  SfRollArgs s = a, r = {};
  s.T = 1;
  r.T = 1; r.flags = a.flags; r.env0 = a.env0; r.envn = a.envn;
  for (int t = 0; t < a.T; t++) {
    const size_t o = (size_t)t * n;  // agent step t alone: its slot of every time-major array
    s.actions = a.actions ? a.actions + o : nullptr; s.t0 = a.t0 + t;
    s.reward = a.reward ? a.reward + o : nullptr; s.done = a.done ? a.done + o : nullptr;
    s.fortkill = a.fortkill ? a.fortkill + o : nullptr; s.events = a.events ? a.events + o : nullptr;
    if (int rc = launch_state(h, s, f, final_mode, t, st)) return rc;
    if (deferred) {  // the finished states into their final-frame slots, then their new games
      r.obs = fo.frames; r.draw_mask = h->d_final_pending;
      if (int rc = launch_draw(h, r, st)) return rc;
      sf_final_reset_kernel<<<(a.envn + SF_STEP_ONLY_BLOCK - 1) / SF_STEP_ONLY_BLOCK, SF_STEP_ONLY_BLOCK, 0, st>>>(h->dev, h->d_final_pending, a.env0, a.envn);
      CUDA_TRY(cudaGetLastError());
      r.draw_mask = nullptr;
    }
    r.obs = a.obs + o * per;
    if (int rc = launch_draw(h, r, st)) return rc;
  }
  return SF_OK;
}

// ------------------------------------------------------------------------------------------------
// policy input (consumer side of the on-device rollout): 4-frame stack -> space-to-depth bf16 NHWC
// ------------------------------------------------------------------------------------------------
#include <cuda_bf16.h>
// One block per env. For each of the 21 output rows Y the 4 frames x 4 pixel rows it needs (1344 B) are staged in
// shared memory with coalesced 32-bit loads (two tiles: one barrier per row), then the 21 x 64 bf16 of the row go out
// as coalesced 16-byte stores (8 channels = frame f, rows dy0, dy0 + 1, 4 columns of block X). u8 -> bf16(u8 / 255)
// through a 256-entry table built with the exact formula (u8 -> fp32, / 255 in fp32, round to bf16, like torch).
#define SF_PI_THREADS 192
template <bool F32>
__global__ void __launch_bounds__(SF_PI_THREADS) sf_policy_input_kernel(const unsigned char* __restrict__ frames, long long fstride, int n, const int* __restrict__ valid,
                                                                       uint4* __restrict__ out) {
  __shared__ unsigned tile[2][4 * 4 * 21];  // [frame][dy][X] : 4 pixels each
  __shared__ unsigned lut[256];             // bf16 bits of u8 / 255 (F32: the fp32 bits)
  const int env = blockIdx.x, tid = threadIdx.x;
  for (int v = tid; v < 256; v += SF_PI_THREADS) {
    // fp32: torch's CUDA `x / 255.0` multiplies by the fp32 reciprocal of the scalar; the table reproduces that bit for bit
    if (F32) lut[v] = __float_as_uint(__fmul_rn((float)v, __fdiv_rn(1.0f, 255.0f)));
    else { const __nv_bfloat16 h = __float2bfloat16_rn(__fdiv_rn((float)v, 255.0f)); lut[v] = *reinterpret_cast<const unsigned short*>(&h); }
  }
  const int nvalid = min(max(valid[env], 0), 4);
  // what this thread loads (words k0 = tid and k1 = tid + 192 of the 336-word tile) and stores (chunk tid < 168)
  const unsigned char* base = frames + (long long)env * (84 * 84);
  const int k1 = tid + SF_PI_THREADS;
  const int f0 = tid / 84, r0 = tid - f0 * 84, f1 = k1 / 84, r1 = k1 - f1 * 84;
  const bool on0 = f0 >= 4 - nvalid, on1 = k1 < 336 && f1 >= 4 - nvalid;
  const unsigned char* p0 = base + (long long)f0 * fstride + (r0 / 21) * 84 + (r0 % 21) * 4;
  const unsigned char* p1 = base + (long long)(k1 < 336 ? f1 : 0) * fstride + (r1 / 21) * 84 + (r1 % 21) * 4;
  const int X = tid >> 3, c8 = tid & 7, f = c8 >> 1, dy0 = (c8 & 1) * 2;
  const int ta = (f * 4 + dy0) * 21 + X, tb = ta + 21;
  uint4* orow = out + (long long)env * (21 * 21 * 8) * (F32 ? 2 : 1);
  auto cvt2 = [&](unsigned lo, unsigned hi) { return lut[lo] | (lut[hi] << 16); };
#pragma unroll 1
  for (int Y = 0; Y < 21; Y++) {
    unsigned* T = tile[Y & 1];
    T[tid] = on0 ? *reinterpret_cast<const unsigned*>(p0 + Y * (4 * 84)) : 0u;
    if (k1 < 336) T[k1] = on1 ? *reinterpret_cast<const unsigned*>(p1 + Y * (4 * 84)) : 0u;
    __syncthreads();  // (the other tile is free again: every thread passed the previous barrier after reading it)
    if (tid < 21 * 8) {
      const unsigned a = T[ta], b = T[tb];
      if (F32) {
        uint4 o0, o1;
        o0.x = lut[a & 255u]; o0.y = lut[(a >> 8) & 255u]; o0.z = lut[(a >> 16) & 255u]; o0.w = lut[a >> 24];
        o1.x = lut[b & 255u]; o1.y = lut[(b >> 8) & 255u]; o1.z = lut[(b >> 16) & 255u]; o1.w = lut[b >> 24];
        orow[(Y * (21 * 8) + tid) * 2] = o0; orow[(Y * (21 * 8) + tid) * 2 + 1] = o1;
      } else {
        uint4 o;
        o.x = cvt2(a & 255u, (a >> 8) & 255u); o.y = cvt2((a >> 16) & 255u, a >> 24);
        o.z = cvt2(b & 255u, (b >> 8) & 255u); o.w = cvt2((b >> 16) & 255u, b >> 24);
        orow[Y * (21 * 8) + tid] = o;
      }
    }
  }
}

static int policy_input_common(const uint8_t* d_frames, long long frame_stride_bytes, int n, const int32_t* d_valid, void* d_out, bool f32, void* stream) {
  if (!d_frames || !d_valid || !d_out || n <= 0 || (frame_stride_bytes & 3)) return fail(SF_ERR_INVALID, "sf_policy_input: bad arguments");
  cudaPointerAttributes pa;  // no handle: launch on the device that owns the frames, whatever the caller's current device is
  CUDA_TRY(cudaPointerGetAttributes(&pa, d_frames));
  if (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) return fail(SF_ERR_INVALID, "sf_policy_input: d_frames is not device memory");
  CUDA_TRY(cudaSetDevice(pa.device));
  if (f32) sf_policy_input_kernel<true><<<(unsigned)n, SF_PI_THREADS, 0, (cudaStream_t)stream>>>(d_frames, frame_stride_bytes, n, d_valid, reinterpret_cast<uint4*>(d_out));
  else sf_policy_input_kernel<false><<<(unsigned)n, SF_PI_THREADS, 0, (cudaStream_t)stream>>>(d_frames, frame_stride_bytes, n, d_valid, reinterpret_cast<uint4*>(d_out));
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}
extern "C" int sf_policy_input(const uint8_t* d_frames, long long frame_stride_bytes, int n, const int32_t* d_valid, void* d_out_bf16, void* stream) {
  return policy_input_common(d_frames, frame_stride_bytes, n, d_valid, d_out_bf16, false, stream);
}
extern "C" int sf_policy_input_f32(const uint8_t* d_frames, long long frame_stride_bytes, int n, const int32_t* d_valid, float* d_out_f32, void* stream) {
  return policy_input_common(d_frames, frame_stride_bytes, n, d_valid, d_out_f32, true, stream);
}

extern "C" int sf_num_features(const sf_handle* h, int obs_type) {
  if (!h) return -1;
  if (obs_type != SF_OBS_FEATURES && obs_type != SF_OBS_NORMALIZED_FEATURES && obs_type != SF_OBS_MONITORS) return -1;
  return sf_feature_cols(h->dev.autoturn, obs_type);
}
static int features_common(sf_handle* h, int obs_type, void* d_out, bool f64, void* stream) {
  if (!h || !d_out) return fail(SF_ERR_INVALID, "handle or out is NULL");
  if (sf_num_features(h, obs_type) < 0) return fail(SF_ERR_INVALID, "obs_type must be SF_OBS_FEATURES, SF_OBS_NORMALIZED_FEATURES or SF_OBS_MONITORS");
  CUDA_TRY(cudaSetDevice(h->device));
  if (f64) sf_features_kernel<double><<<(h->dev.n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->dev, obs_type, (double*)d_out);
  else sf_features_kernel<float><<<(h->dev.n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->dev, obs_type, (float*)d_out);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}
extern "C" int sf_features(sf_handle* h, int obs_type, float* d_out, void* stream) { return features_common(h, obs_type, d_out, false, stream); }
extern "C" int sf_features_f64(sf_handle* h, int obs_type, double* d_out, void* stream) { return features_common(h, obs_type, d_out, true, stream); }

extern "C" int sf_set_ticks(sf_handle* h, const int32_t* h_ticks) {
  if (!h || !h_ticks) return fail(SF_ERR_INVALID, "handle or ticks is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  int* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(int) * (size_t)h->dev.n));
  cudaError_t ce = cudaDeviceSynchronize();  // synchronous call: ordered after whatever any stream has queued for this slab
  if (ce == cudaSuccess) ce = cudaMemcpy(d, h_ticks, sizeof(int) * (size_t)h->dev.n, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) {
    sf_set_ticks_kernel<<<(h->dev.n + 127) / 128, 128>>>(h->dev, d);
    ce = cudaDeviceSynchronize();
  }
  cudaFree(d);
  if (ce != cudaSuccess) return fail(SF_ERR_CUDA, std::string("sf_set_ticks: ") + cudaGetErrorString(ce));
  return SF_OK;
}

extern "C" int sf_reset(sf_handle* h, const uint8_t* d_mask, int clear_prev_vlner, uint8_t* d_obs, int flags, void* stream) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  sf_reset_kernel<<<(h->dev.n + 127) / 128, 128, 0, st>>>(h->dev, d_mask, clear_prev_vlner);
  CUDA_TRY(cudaGetLastError());
  if (!d_obs) return SF_OK;
  SfRollArgs a = {};
  a.T = 1; a.obs = d_obs; a.flags = flags | SF_FLAG_RENDER; a.envn = h->dev.n; a.draw_mask = d_mask;
  return launch_draw(h, a, st);
}

extern "C" int sf_render(sf_handle* h, uint8_t* d_obs, int flags, void* stream) {
  if (!h || !d_obs) return fail(SF_ERR_INVALID, "handle or obs is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  SfRollArgs a = {};
  a.T = 1; a.obs = d_obs; a.flags = flags | SF_FLAG_RENDER; a.envn = h->dev.n;
  return launch_draw(h, a, (cudaStream_t)stream);
}

extern "C" int sf_step(sf_handle* h, const int32_t* d_actions, uint8_t* d_obs, int32_t* d_reward, uint8_t* d_done,
                       uint8_t* d_fortkill, uint32_t* d_events, int flags, void* stream) {
  if (!h || !d_actions) return fail(SF_ERR_INVALID, "handle or actions is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  SfRollArgs a = {};
  a.T = 1; a.flags = flags; a.actions = d_actions;
  a.obs = d_obs; a.reward = d_reward; a.done = d_done; a.fortkill = d_fortkill; a.events = d_events; a.envn = h->dev.n;
  return launch_steps(h, a, {}, (cudaStream_t)stream);
}

extern "C" int sf_rollout(sf_handle* h, int T, const int32_t* d_actions, uint32_t action_seed, long long t0, uint8_t* d_obs,
                          int32_t* d_reward, uint8_t* d_done, uint8_t* d_fortkill, int flags, void* stream) {
  if (!h || T <= 0) return fail(SF_ERR_INVALID, "handle is NULL or T <= 0");
  CUDA_TRY(cudaSetDevice(h->device));
  SfRollArgs a = {};
  a.T = T; a.flags = flags; a.actions = d_actions; a.action_seed = action_seed; a.t0 = t0;
  a.obs = d_obs; a.reward = d_reward; a.done = d_done; a.fortkill = d_fortkill; a.envn = h->dev.n;
  return launch_steps(h, a, {}, (cudaStream_t)stream);
}

// the checks both feature steps share; *nf = the row width
static int feature_step_args(const sf_handle* h, int obs_type, const float* features, int flags, int* nf) {
  if (!h || !features) return fail(SF_ERR_INVALID, "handle or features is NULL");
  if ((*nf = sf_num_features(h, obs_type)) < 0) return fail(SF_ERR_INVALID, "obs_type must be SF_OBS_FEATURES, SF_OBS_NORMALIZED_FEATURES or SF_OBS_MONITORS");
  if (flags & (SF_FLAG_RENDER | SF_FLAG_NATIVE_OBS | SF_FLAG_HOST_DELTA))
    return fail(SF_ERR_INVALID, "a feature step draws no frames: SF_FLAG_RENDER, SF_FLAG_NATIVE_OBS and SF_FLAG_HOST_DELTA are invalid");
  return SF_OK;
}

extern "C" int sf_rollout_features(sf_handle* h, int obs_type, int T, const int32_t* d_actions, uint32_t action_seed, long long t0,
                                   float* d_features, int32_t* d_reward, uint8_t* d_done, uint8_t* d_fortkill, uint32_t* d_events,
                                   int flags, void* stream) {
  int nf;
  if (int rc = feature_step_args(h, obs_type, d_features, flags, &nf)) return rc;
  if (T <= 0) return fail(SF_ERR_INVALID, "T <= 0");
  CUDA_TRY(cudaSetDevice(h->device));
  SfRollArgs a = {};
  a.T = T; a.flags = flags; a.actions = d_actions; a.action_seed = action_seed; a.t0 = t0;
  a.reward = d_reward; a.done = d_done; a.fortkill = d_fortkill; a.events = d_events; a.envn = h->dev.n;
  return launch_steps(h, a, SfFeatArgs{d_features, obs_type, nf}, (cudaStream_t)stream);
}

extern "C" int sf_set_action_repeat(sf_handle* h, int k) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  if (k < 1 || k > SF_MAX_ACTION_REPEAT) return fail(SF_ERR_INVALID, "action repeat must be in [1, " + std::to_string(SF_MAX_ACTION_REPEAT) + "]");
  h->action_repeat = k;
  return SF_OK;
}
extern "C" int sf_action_repeat(const sf_handle* h) { return h ? h->action_repeat : -1; }

static bool sticky_p_ok(double p) { return p >= 0.0 && p <= 1.0; }  // false for NaN
static unsigned long long sticky_threshold(double p) { return (unsigned long long)std::llround(p * 4294967296.0); }
extern "C" int sf_set_sticky_actions(sf_handle* h, double p, uint32_t seed) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  if (!sticky_p_ok(p)) return fail(SF_ERR_INVALID, "repeat_action_probability must be in [0, 1]");
  h->sticky_p = p;
  h->sticky = SfStickyArgs{sticky_threshold(p), seed};
  return SF_OK;
}
extern "C" double sf_sticky_actions(const sf_handle* h) { return h ? h->sticky_p : -1.0; }
extern "C" int sf_sticky_draw(uint32_t seed, long long global_env, uint32_t rng_count, int32_t tick, double p) {
  if (!sticky_p_ok(p)) return fail(-1, "repeat_action_probability must be in [0, 1]");
  return sf_sticky_hash(seed, (unsigned long long)global_env, rng_count, tick, sticky_threshold(p)) ? 1 : 0;
}

extern "C" int sf_set_final_obs(sf_handle* h, uint8_t* d_frames, float* d_rows, int32_t* d_final_step) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  if ((d_frames || d_rows) && !d_final_step) return fail(SF_ERR_INVALID, "final observations need d_final_step");
  if (d_final_step && !h->d_final_pending) {
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMalloc(&h->d_final_pending, (size_t)h->dev.n));
    CUDA_TRY(cudaMemset(h->d_final_pending, 0, (size_t)h->dev.n));
  }
  h->final_obs = sf_handle::FinalObs{d_frames, d_rows, d_final_step};
  return SF_OK;
}
extern "C" int sf_final_obs_enabled(const sf_handle* h) { return h ? (h->final_obs.step != nullptr) : -1; }

extern "C" int sf_synthetic_action(uint32_t action_seed, long long global_env, long long t, int num_actions) {
  return sf_hash_action(action_seed, (unsigned long long)global_env, (unsigned long long)t, num_actions);
}

static int ensure_staging(sf_handle* h, size_t obs_bytes) {
  size_t n = (size_t)h->dev.n;
  if (!h->host_compute) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->host_compute, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&h->host_copy, cudaStreamNonBlocking));
    for (int k = 0; k < SF_HOST_STEP_SLICES; k++) CUDA_TRY(cudaEventCreateWithFlags(&h->host_ev[k], cudaEventDisableTiming));
  }
  if (!h->d_actions) {
    CUDA_TRY(cudaMalloc(&h->d_actions, n * 4)); CUDA_TRY(cudaMalloc(&h->d_reward, n * 4));
    CUDA_TRY(cudaMalloc(&h->d_done, n)); CUDA_TRY(cudaMalloc(&h->d_kill, n)); CUDA_TRY(cudaMalloc(&h->d_events, n * 4));
  }
  if (obs_bytes > h->staging_obs_bytes) {
    if (h->d_obs) { cudaFree(h->d_obs); h->d_obs = nullptr; }
    CUDA_TRY(cudaMalloc(&h->d_obs, obs_bytes));
    h->staging_obs_bytes = obs_bytes;
  }
  return SF_OK;
}

extern "C" int sf_host_alloc(void** out, long long bytes) {
  if (!out || bytes <= 0) return fail(SF_ERR_INVALID, "sf_host_alloc: bad arguments");
  CUDA_TRY(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable | cudaHostAllocMapped));
  return SF_OK;
}
extern "C" int sf_host_free(void* p) {
  if (p) CUDA_TRY(cudaFreeHost(p));
  return SF_OK;
}

// The device's address for a page-locked host buffer (NULL for pageable memory): kernels read / write such buffers in
// place across PCIe, which for the small per-env arrays of a step replaces a DMA copy (several microseconds each).
static void* device_alias(const void* host) {
  cudaPointerAttributes at;
  if (!host || cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

// sf_step_host and sf_step_host_features. h_feat (frames off): feature rows of kind feat_kind, nfeat floats each.
static int step_host(sf_handle* h, const int32_t* h_actions, uint8_t* h_obs, float* h_feat, int feat_kind, int nfeat, int32_t* h_reward,
                     uint8_t* h_done, uint8_t* h_fortkill, uint32_t* h_events, int flags) {
  if (!h || !h_actions) return fail(SF_ERR_INVALID, "handle or actions is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t n = (size_t)h->dev.n;
  const size_t per = (flags & SF_FLAG_NATIVE_OBS) ? (size_t)SF_NAT_H * SF_NAT_W : (size_t)84 * 84, obs_bytes = n * per;
  const bool render = (flags & SF_FLAG_RENDER) && h_obs;
  // page-locked feature rows are written in place like the small arrays below; pageable ones go through the obs staging
  float* k_feat = (float*)device_alias(h_feat);
  const size_t feat_bytes = n * nfeat * sizeof(float);
  int rc = ensure_staging(h, render ? obs_bytes : (h_feat && !k_feat) ? feat_bytes : 0);
  if (rc) return rc;
  // Synchronous, on the handle's own streams. Whole-frame mode: the slab is stepped in slices of consecutive envs, the
  // kernel of slice k + 1 runs while the frames of slice k cross PCIe (one cudaMemcpyAsync per buffer and slice), so only
  // the first slice's kernel is exposed. Delta mode: one launch, no copies (see sf_block_host_delta). Work the caller has
  // queued on OTHER streams for this handle must be complete (the Python wrapper synchronises its stream first);
  // everything queued here is complete on return.
  cudaStream_t sc = h->host_compute, sx = h->host_copy;
  // SF_FLAG_HOST_DELTA: h_obs is page-locked and still holds what the previous call with this flag wrote there
  uint4* host_alias = nullptr;
  sf_handle::Mirror* mir = nullptr;
  const bool want_delta = render && (flags & SF_FLAG_HOST_DELTA);
  if (want_delta) {
    host_alias = reinterpret_cast<uint4*>(device_alias(h_obs));
    if (!host_alias) return fail(SF_ERR_INVALID, "SF_FLAG_HOST_DELTA needs a page-locked h_obs (sf_host_alloc, cudaHostAlloc, cudaHostRegister)");
    if (((uintptr_t)h_obs | (uintptr_t)host_alias) & 15) return fail(SF_ERR_INVALID, "SF_FLAG_HOST_DELTA needs a 16-byte aligned h_obs");
    if ((rc = h->mirror_for(h_obs, obs_bytes, &mir))) return rc;
    if (!h->d_delta_stats) {
      CUDA_TRY(cudaMalloc(&h->d_delta_stats, 16));
      CUDA_TRY(cudaMemset(h->d_delta_stats, 0, 16));
    }
  }
  const bool delta = want_delta && mir->host == h_obs && mir->bytes == obs_bytes;
  // the blocks of the fused kernel send their own frames' changes (split frames come from draw launches)
  const bool fused_delta = delta && per % 16 == 0 && !frames_need_split(h);
  CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));  // calls made with stream == NULL (sf_reset, sf_seed ...) come first
  // page-locked actions / rewards / dones / kills / events are read and written in place by the kernel
  const int* k_actions = (const int*)device_alias(h_actions);
  int* k_reward = (int*)device_alias(h_reward);
  unsigned char* k_done = (unsigned char*)device_alias(h_done);
  unsigned char* k_kill = (unsigned char*)device_alias(h_fortkill);
  unsigned* k_events = (unsigned*)device_alias(h_events);
  if (!k_actions) CUDA_TRY(cudaMemcpyAsync(h->d_actions, h_actions, n * 4, cudaMemcpyHostToDevice, sc));
  flags &= ~SF_FLAG_HOST_DELTA;
  SfRollArgs a = {};
  a.T = 1; a.flags = render ? flags : (flags & ~SF_FLAG_RENDER);
  a.actions = k_actions ? k_actions : h->d_actions;
  a.obs = render ? h->d_obs : nullptr; a.reward = k_reward ? k_reward : h->d_reward; a.done = k_done ? k_done : h->d_done;
  a.fortkill = k_kill ? k_kill : h->d_kill; a.events = k_events ? k_events : h->d_events;
  if (fused_delta) { a.host_obs = host_alias; a.mirror = reinterpret_cast<uint4*>(mir->d); a.delta_stats = h->d_delta_stats; }
  const SfFeatArgs f = {h_feat ? (k_feat ? k_feat : reinterpret_cast<float*>(h->d_obs)) : nullptr, feat_kind, nfeat};
  const int slices = (render && !delta && n >= 2048) ? SF_HOST_STEP_SLICES : 1;
  for (int k = 0; k < slices; k++) {
    const size_t e0 = n * k / slices, e1 = n * (k + 1) / slices;
    a.env0 = (int)e0; a.envn = (int)(e1 - e0);
    rc = launch_steps(h, a, f, sc);
    if (rc) { cudaStreamSynchronize(sc); cudaStreamSynchronize(sx); return rc; }
    if (render && !delta) {
      CUDA_TRY(cudaEventRecord(h->host_ev[k], sc));
      CUDA_TRY(cudaStreamWaitEvent(sx, h->host_ev[k], 0));
      CUDA_TRY(cudaMemcpyAsync(h_obs + e0 * per, h->d_obs + e0 * per, (e1 - e0) * per, cudaMemcpyDeviceToHost, sx));
    }
  }
  if (delta && !fused_delta) {
    const size_t n16 = obs_bytes / 16;
    const int blocks = (int)std::min<size_t>((n16 + 255) / 256, (size_t)h->num_sms * 8);
    sf_host_delta_kernel<<<std::max(blocks, 1), 256, 0, sc>>>(reinterpret_cast<const uint4*>(h->d_obs), reinterpret_cast<uint4*>(mir->d), host_alias,
                                                              n16, (int)(obs_bytes & 15), h->d_delta_stats);
    CUDA_TRY(cudaGetLastError());
  } else if (want_delta) {  // whole frames went out: from here on the mirror describes this buffer
    CUDA_TRY(cudaMemcpyAsync(mir->d, h->d_obs, obs_bytes, cudaMemcpyDeviceToDevice, sc));
    mir->host = h_obs; mir->bytes = obs_bytes;
  }
  if (render && !delta) h->full_calls++;
  if (h_feat && !k_feat) CUDA_TRY(cudaMemcpyAsync(h_feat, h->d_obs, feat_bytes, cudaMemcpyDeviceToHost, sc));
  if (h_reward && !k_reward) CUDA_TRY(cudaMemcpyAsync(h_reward, h->d_reward, n * 4, cudaMemcpyDeviceToHost, sc));
  if (h_done && !k_done) CUDA_TRY(cudaMemcpyAsync(h_done, h->d_done, n, cudaMemcpyDeviceToHost, sc));
  if (h_fortkill && !k_kill) CUDA_TRY(cudaMemcpyAsync(h_fortkill, h->d_kill, n, cudaMemcpyDeviceToHost, sc));
  if (h_events && !k_events) CUDA_TRY(cudaMemcpyAsync(h_events, h->d_events, n * 4, cudaMemcpyDeviceToHost, sc));
  cudaError_t e1 = cudaStreamSynchronize(sc), e2 = (render && !delta) ? cudaStreamSynchronize(sx) : cudaSuccess;
  if (e1 != cudaSuccess || e2 != cudaSuccess) {
    h->forget_mirrors(nullptr);
    return fail(SF_ERR_CUDA, std::string("sf_step_host: ") + cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  }
  return SF_OK;
}

extern "C" int sf_step_host(sf_handle* h, const int32_t* h_actions, uint8_t* h_obs, int32_t* h_reward, uint8_t* h_done,
                            uint8_t* h_fortkill, uint32_t* h_events, int flags) {
  return step_host(h, h_actions, h_obs, nullptr, 0, 0, h_reward, h_done, h_fortkill, h_events, flags);
}

extern "C" int sf_step_host_features(sf_handle* h, int obs_type, const int32_t* h_actions, float* h_features, int32_t* h_reward,
                                     uint8_t* h_done, uint8_t* h_fortkill, uint32_t* h_events, int flags) {
  int nf;
  if (int rc = feature_step_args(h, obs_type, h_features, flags, &nf)) return rc;
  return step_host(h, h_actions, nullptr, h_features, obs_type, nf, h_reward, h_done, h_fortkill, h_events, flags);
}

extern "C" int sf_host_forget(sf_handle* h, const void* h_obs) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  h->forget_mirrors(h_obs);
  return SF_OK;
}

extern "C" int sf_host_delta_stats(sf_handle* h, unsigned long long* out3) {
  if (!h || !out3) return fail(SF_ERR_INVALID, "handle or out is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  out3[0] = out3[1] = 0; out3[2] = h->full_calls;
  if (h->d_delta_stats) {
    CUDA_TRY(cudaStreamSynchronize(h->host_compute));
    CUDA_TRY(cudaMemcpy(out3, h->d_delta_stats, 16, cudaMemcpyDeviceToHost));
  }
  return SF_OK;
}

extern "C" int sf_get_state(sf_handle* h, int first, int count, sf_state_record* h_out) {
  if (!h || !h_out || first < 0 || count < 0 || first + count > h->dev.n) return fail(SF_ERR_INVALID, "bad range");
  if (count == 0) return SF_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  sf_state_record* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(sf_state_record) * (size_t)count));
  cudaError_t ce = cudaDeviceSynchronize();  // every stream: the state may be in flight on the caller's stream
  if (ce == cudaSuccess) {
    sf_get_state_kernel<<<(count + 63) / 64, 64>>>(h->dev, first, count, d);
    ce = cudaMemcpy(h_out, d, sizeof(sf_state_record) * (size_t)count, cudaMemcpyDeviceToHost);
  }
  cudaFree(d);
  if (ce != cudaSuccess) return fail(SF_ERR_CUDA, std::string("get_state: ") + cudaGetErrorString(ce));
  return SF_OK;
}

extern "C" int sf_set_state(sf_handle* h, int first, int count, const sf_state_record* h_in) {
  if (!h || !h_in || first < 0 || count < 0 || first + count > h->dev.n) return fail(SF_ERR_INVALID, "bad range");
  for (int k = 0; k < count; k++) {
    const sf_state_record& r = h_in[k];
    if (r.ship_angle != (double)(int)r.ship_angle || r.ship_angle < 0 || r.ship_angle >= 360)
      return fail(SF_ERR_UNSUPPORTED, "ship_angle must be an integer degree in [0,360) (it always is in the reference: game.cpp:148,317-324)");
    double fa = r.fortress_angle / 10.0, fl = r.fortress_last_angle / 10.0;
    if (fa != (double)(int)fa || fa < 0 || fa >= 36 || fl != (double)(int)fl || fl < 0 || fl >= 36)
      return fail(SF_ERR_UNSUPPORTED, "fortress angles must be multiples of 10 in [0,360) (game.cpp:40-41,206)");
    if (r.shell_mask >> SF_DEV_SHELLS) return fail(SF_ERR_UNSUPPORTED, "shell slots >= 4 can never be alive (at most 3 shells are in flight)");
    if (r.missile_mask >> SF_MAX_MISSILES) return fail(SF_ERR_INVALID, "missile_mask has more than 20 bits");
    for (int s = 0; s < SF_MAX_MISSILES; s++) if ((r.missile_mask >> s) & 1) {
      double a = r.missile_angle[s];
      if (a != (double)(int)a || a < 0 || a >= 360) return fail(SF_ERR_UNSUPPORTED, "missile angles must be integer degrees in [0,360)");
    }
  }
  if (count == 0) return SF_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  sf_state_record* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(sf_state_record) * (size_t)count));
  cudaError_t ce = cudaMemcpy(d, h_in, sizeof(sf_state_record) * (size_t)count, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
  if (ce == cudaSuccess) {
    sf_set_state_kernel<<<(count + 63) / 64, 64>>>(h->dev, first, count, d);
    ce = cudaDeviceSynchronize();
  }
  cudaFree(d);
  if (ce != cudaSuccess) return fail(SF_ERR_CUDA, std::string("set_state: ") + cudaGetErrorString(ce));
  return SF_OK;
}

static int blob_args(const sf_handle* h, const int32_t* d_env_idx, int count, const void* d_blob) {
  if (!h || !d_blob) return fail(SF_ERR_INVALID, "handle or blob is NULL");
  if (count < 0 || (!d_env_idx && count > h->dev.n)) return fail(SF_ERR_INVALID, "count out of range");
  if ((uintptr_t)d_blob & 15) return fail(SF_ERR_INVALID, "the blob must be 16-byte aligned");
  return SF_OK;
}
static int blob_blocks(const sf_handle* h, int count) { return std::min((count + 31) / 32, h->num_sms * SF_BLOB_BLOCKS_PER_SM); }

extern "C" int sf_save_envs(sf_handle* h, const int32_t* d_env_idx, int count, uint8_t* d_blob, void* stream) {
  if (int rc = blob_args(h, d_env_idx, count, d_blob)) return rc;
  if (count == 0) return SF_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  sf_save_envs_kernel<<<blob_blocks(h, count), 32, 0, (cudaStream_t)stream>>>(h->dev, h->gametype, d_env_idx, count, reinterpret_cast<int4*>(d_blob));
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_load_envs(sf_handle* h, const uint8_t* d_blob, const int32_t* d_env_idx, int count, int32_t* d_rejected, void* stream) {
  if (int rc = blob_args(h, d_env_idx, count, d_blob)) return rc;
  if (count == 0) return SF_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  sf_load_envs_kernel<<<blob_blocks(h, count), 32, 0, (cudaStream_t)stream>>>(h->dev, h->gametype, reinterpret_cast<const int4*>(d_blob), d_env_idx, count, d_rejected);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

__global__ void sf_epi_copy_kernel(unsigned long long* epi, long long* out, int reset) {
  int k = threadIdx.x;
  if (k < SF_NUM_EPISODE_STATS) {
    out[k] = (long long)epi[k];
    if (reset) epi[k] = 0;
  }
}

extern "C" int sf_episode_stats(sf_handle* h, long long* d_out, int reset, void* stream) {
  if (!h || !d_out) return fail(SF_ERR_INVALID, "handle or out is NULL");
  CUDA_TRY(cudaSetDevice(h->device));
  sf_epi_copy_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->dev.epi, d_out, reset);
  CUDA_TRY(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_set_glyph_masks(sf_handle* h, const uint8_t* h_alpha, const uint8_t* h_slot) {
  if (!h || (!h_alpha) != (!h_slot)) return fail(SF_ERR_INVALID, "handle is NULL, or only one of alpha / slot given");
  SfTables* nt = new SfTables();
  char err[256] = {0};
  if (sf_build_tables_glyphs(nt, err, sizeof(err), h_alpha, h_slot)) { std::string m = err; delete nt; return fail(SF_ERR_INVALID, "table build failed: " + m); }
  cudaError_t ce = cudaSetDevice(h->device);
  if (ce == cudaSuccess) ce = cudaDeviceSynchronize();  // nothing may be drawing from the old tables
  if (ce == cudaSuccess) ce = cudaMemcpy((void*)h->dev.tab, nt, sizeof(SfTables), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemset(h->dev.expo_meta, 0, sizeof(uint2) * (size_t)h->dev.n_pad);  // cached resampled boxes may hold old digits
  if (ce == cudaSuccess) {
    sf_pack_static_kernel<<<1, SF_BLOCK, SF_RENDER_SMEM_BYTES(SF_RENDER_WARPS)>>>(h->dev, const_cast<unsigned char*>(h->dev.static_image));
    ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
  }
  if (ce != cudaSuccess) { delete nt; return fail(SF_ERR_CUDA, std::string("sf_set_glyph_masks: ") + cudaGetErrorString(ce)); }
  delete h->h_tab;
  h->h_tab = nt;
  return SF_OK;
}

extern "C" int sf_background(const sf_handle* h, uint8_t* h_native, uint8_t* h_obs) {
  if (!h) return fail(SF_ERR_INVALID, "handle is NULL");
  if (h_native)
    for (int r = 0; r < SF_NAT_H; r++) memcpy(h_native + r * SF_NAT_W, h->h_tab->bg_nat + r * SF_NAT_STRIDE, SF_NAT_W);
  if (h_obs) memcpy(h_obs, h->h_tab->bg_obs, 84 * 84);
  return SF_OK;
}
