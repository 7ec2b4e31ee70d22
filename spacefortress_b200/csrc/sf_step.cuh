// sf_step.cuh — one game tick + env shaping + auto-reset for ONE env, executed by one thread.
// Replaces Game::stepOneTick (game.cpp:473-485) and SSF_Env.step's reward/done logic
// (ssf_env.py:208-253). Integer state and events are bit-exact against the reference; fp64
// kinematics use explicit round-to-nearest single operations (the reference is built without FMA
// contraction), integer-degree trig comes from a host-libm LUT, and the only device transcendentals
// are atan2 (aiming, quantised by ceil) and cos/sin of the real-valued shell angle.
#pragma once
#include "sf_geom.h"
#include "sf_state.cuh"
#include "../../include/sf_b200.h"
#include "sf_probe.cuh"

#define SF_TICK_MS 34        // ssf_env.py:61
#define SF_GAME_TIME 180000  // configs.cpp:55,66,78,86
#define SF_GAME_TICKS 5295   // first tick with mTime >= gameTime (game.cpp:487-489)

struct SfStepOut {
  int reward;       // shaped (train presets) or raw (test presets) integer reward
  unsigned events;  // SF_EV_*
  bool done, fort_kill;
  unsigned shell_vis;  // live shells further than 21 from the fortress after the tick (what draw.cpp:249-250 shows), bit per slot
};

// Registers of one env between load and store. The twelve Stats counters of st0..st2 (game.hh:29-43) change on a few
// ticks only, so the step does not carry them: it counts the tick's increments in three words of four 8-bit fields
// (d0 / d1 / d2 line up with the components of st0 / st1 / st2) and sf_store_env adds them to the arrays only when one is
// non-zero. That is 96 B less traffic per env-step and 9 registers less for the step.
struct SfEnv {
  double2 pos, vel;
  int4 q0, q1, q2, q3, st3;
  unsigned d0, d1, d2;   // pending increments: st0 (bigHexDeaths smallHexDeaths shellDeaths shipDeaths), st1 (resets destroyedFortresses missedShots totalShots), st2 (totalThrusts totalLefts totalRights vlnerIncs)
};
#define SF_ST_INC(word, comp) ((word) += 1u << (8 * (comp)))

__device__ __forceinline__ void sf_load_env(const SfDev& D, int i, SfEnv& e) {
  e.pos = D.pos[i]; e.vel = D.vel[i];
  e.q0 = D.q0[i]; e.q1 = D.q1[i]; e.q2 = D.q2[i]; e.q3 = D.q3[i];
  e.st3 = D.st3[i];
  e.d0 = 0u; e.d1 = 0u; e.d2 = 0u;
}
// the pending Stats increments -> the arrays (a field holds up to 255: flush at least every 12 ticks — 20 missiles could
// leave the area in one tick)
// (Reductions, not load-add-store: the stepping warp is bound by latency, and a reduction does not wait for the memory.
// Only this lane ever touches env i's counters, so the atomicity itself is not needed.)
__device__ __forceinline__ void sf_red_bytes(int4* p, unsigned d) {
  int* q = reinterpret_cast<int*>(p);
  if (d & 0x000000FFu) atomicAdd(q + 0, (int)(d & 255u));
  if (d & 0x0000FF00u) atomicAdd(q + 1, (int)((d >> 8) & 255u));
  if (d & 0x00FF0000u) atomicAdd(q + 2, (int)((d >> 16) & 255u));
  if (d & 0xFF000000u) atomicAdd(q + 3, (int)(d >> 24));
}
__device__ __forceinline__ void sf_flush_stats(const SfDev& D, int i, SfEnv& e) {
  if (e.d0) { sf_red_bytes(&D.st0[i], e.d0); e.d0 = 0u; }
  if (e.d1) { sf_red_bytes(&D.st1[i], e.d1); e.d1 = 0u; }
  if (e.d2) { sf_red_bytes(&D.st2[i], e.d2); e.d2 = 0u; }
}
__device__ __forceinline__ void sf_store_env(const SfDev& D, int i, SfEnv& e) {
  D.pos[i] = e.pos; D.vel[i] = e.vel;
  D.q0[i] = e.q0; D.q1[i] = e.q1; D.q2[i] = e.q2; D.q3[i] = e.q3;
  D.st3[i] = e.st3;
  sf_flush_stats(D, i, e);
}

// ---- G1: glibc rand() (TYPE_3 lagged sum over a 31-word ring), one stream per env ----
__device__ __forceinline__ int sf_rand_raw(unsigned* rng, int np, int i, int& idx) {
  int lag = idx + 28; if (lag >= 31) lag -= 31;  // (k-3) mod 31
  unsigned v = rng[(size_t)idx * np + i] + rng[(size_t)lag * np + i];
  rng[(size_t)idx * np + i] = v;
  idx = (idx + 1 == 31) ? 0 : idx + 1;
  return (int)(v >> 1);
}
__device__ __forceinline__ int sf_rand(const SfDev& D, int i, SfEnv& e) {
  int idx = e.st3.y;
  int r = sf_rand_raw(D.rng, D.n_pad, i, idx);
  e.st3.y = idx; e.st3.z += 1;
  return r;
}

// srand(seed): r[0]=seed, r[k]=16807*r[k-1] mod (2^31-1), 310 outputs dropped
__device__ inline void sf_srand(const SfDev& D, int i, SfEnv& e, unsigned seed) {
  if (seed == 0) seed = 1;
  int w = (int)seed;
  D.rng[i] = (unsigned)w;
  for (int k = 1; k < 31; k++) {
    long long hi = w / 127773, lo = w % 127773;
    long long v = 16807 * lo - 2836 * hi;
    if (v < 0) v += 2147483647;
    w = (int)v;
    D.rng[(size_t)k * D.n_pad + i] = (unsigned)w;
  }
  e.st3.y = 3;  // 34 mod 31
  for (int k = 0; k < 310; k++) (void)sf_rand(D, i, e);
  e.st3.z = 0;
  e.st3.w = (int)seed;
}

// ---- S9: Hexagon::isInside (hexagon.cpp:37-48), boundary inclusive ----
__device__ __forceinline__ bool sf_inside_hex(const SfHot* H, int h, double x, double y) {
  bool in = true;
#pragma unroll
  for (int k = 0; k < 6; k++) {
    double dx = SF_DSUB(x, H->hex[h][k][0]), dy = SF_DSUB(y, H->hex[h][k][1]);
    double t = SF_DADD(SF_DMUL(H->hex[h][k][2], dx), SF_DMUL(H->hex[h][k][3], dy));
    in = in && !(t < 0);
  }
  return in;
}

// object.cpp:12-15: sqrt(dx*dx + dy*dy) <= r, evaluated without the square root as d2 <= T(r) (SfHot::touch2: the
// same decision for every double d2, checked on the host)
__device__ __forceinline__ double sf_dist2(double ax, double ay, double bx, double by) {
  double dx = SF_DSUB(ax, bx), dy = SF_DSUB(ay, by);
  return SF_DADD(SF_DMUL(dx, dx), SF_DMUL(dy, dy));
}
__device__ __forceinline__ bool sf_outside(double x, double y) {  // game.cpp:129-131
  return x < 0 || x > 710.0 || y > 626.0 || y < 0;
}

// atan2 as the reference's libm gives it where a downstream ceil() could flip (exact octants);
// elsewhere the CUDA fp64 atan2 (<= 2 ulp) is used — a differing last bit cannot change the
// quantised angle unless the true angle is within 1e-13 degrees of an integer.
__device__ __noinline__ double sf_atan2(const SfHot* H, double dy, double dx) {
  if (dy == 0.0) return dx >= 0 ? H->atan2_oct[0] : H->atan2_oct[4];
  if (dx == 0.0) return dy > 0 ? H->atan2_oct[2] : H->atan2_oct[6];
  if (fabs(dx) == fabs(dy)) return dx > 0 ? (dy > 0 ? H->atan2_oct[1] : H->atan2_oct[7]) : (dy > 0 ? H->atan2_oct[3] : H->atan2_oct[5]);
  return atan2(dy, dx);
}
#define SF_PI 3.14159265358979323846
__device__ __forceinline__ double sf_rad2deg(double a) { return SF_DMUL(SF_DDIV(a, SF_PI), 180.0); }  // vector.cpp:38-40
__device__ __forceinline__ double sf_deg2rad(double a) { return SF_DDIV(SF_DMUL(a, SF_PI), 180.0); }  // vector.cpp:34-36

// The reference quantises both of its aiming angles with ceil(): the autoturn heading ceil(angleTo(ship, fortress))
// (game.cpp:319, vector.cpp:48-52) and the fortress sector ceil(angle_to_ship / 10) * 10 (game.cpp:197,206). Only the
// smallest multiple k of STEP degrees with k >= theta matters, theta in [0, 360) being the direction of (dx, dy). That
// is a sign test, not a transcendental: theta <= k  <=>  sin(theta - k) <= 0  <=>  cos(k) * dy - sin(k) * dx <= 0, with
// cos / sin of integer degrees from the host-libm table. An fp32 atan2f proposes k (within one STEP of the answer), two
// fp64 cross products confirm or move it. It decides like ceil(rad2deg(atan2())) unless theta lies within ~1e-14
// degrees of a multiple of STEP — the same measure-zero band in which the 2-ulp device atan2 used before could differ
// from libm — and the exact octants (the only directions with integer coordinates that ARE multiples of STEP) go through
// the reference's own libm values (sf_atan2) and its own operation order.
__device__ __noinline__ int sf_ceil_angle_exact(const SfHot* H, double dy, double dx, int step, bool add_before) {
  double deg;
  if (add_before) {  // angleTo (vector.cpp:48-52): a < 0 -> a += 2 pi, then rad2deg
    double a = sf_atan2(H, dy, dx);
    if (a < 0) a = SF_DADD(a, SF_PI * 2);
    deg = sf_rad2deg(a);
  } else {           // updateFortress (game.cpp:197): stdAngle(rad2deg(a))
    deg = sf_rad2deg(sf_atan2(H, dy, dx));
    if (deg < 0) deg = SF_DADD(deg, 360.0);
  }
  return step * (int)ceil(SF_DDIV(deg, (double)step));
}
template <int STEP>
__device__ __forceinline__ int sf_ceil_angle(const SfHot* H, double dy, double dx, bool add_before) {  // in [0, 360]
  if (dy == 0.0 || dx == 0.0 || fabs(dx) == fabs(dy)) return sf_ceil_angle_exact(H, dy, dx, STEP, add_before);
  float a = atan2f((float)dy, (float)dx) * 57.29577951308232f;
  if (a < 0.f) a += 360.f;
  int k = STEP * (int)ceilf(a * (1.0f / STEP));
  k = min(max(k, STEP), 360);
  const int ik = k == 360 ? 0 : k, im = k - STEP;
  const double fk = SF_DSUB(SF_DMUL(H->cs[ik][0], dy), SF_DMUL(H->cs[ik][1], dx));
  const double fm = SF_DSUB(SF_DMUL(H->cs[im][0], dy), SF_DMUL(H->cs[im][1], dx));
  if (fk > 0) k += STEP;          // theta > k
  else if (fm <= 0) k -= STEP;    // theta <= k - STEP
  return k;
}

// S12: shell velocity 6*(cos,sin)(deg2rad(angle)) for a real-valued angle (game.cpp:167-168); out of line: rare
__device__ __noinline__ double2 sf_shell_velocity(double a) {
  double rad = sf_deg2rad(a);
  return make_double2(SF_DMUL(6.0, cos(rad)), SF_DMUL(6.0, sin(rad)));
}

// S15: reward()/penalize() in float32 (game.cpp:97-106)
__device__ __forceinline__ void sf_reward(SfEnv& e, float& tick_reward, float amt) {
  tick_reward = __fadd_rn(tick_reward, amt);
  float raw = __fadd_rn(__int_as_float(e.q3.y), amt);
  float pts = __fadd_rn(__int_as_float(e.q3.x), amt);
  if (pts < 0) pts = 0;
  e.q3.x = __float_as_int(pts); e.q3.y = __float_as_int(raw);
}

__device__ __forceinline__ void sf_kill_ship(SfEnv& e) {  // game.cpp:274-280
  if (e.q0.x & SF_CORE_SHIP_ALIVE) {
    e.q0.x &= ~SF_CORE_SHIP_ALIVE;
    e.q0.z = 0;
    SF_ST_INC(e.d0, 3);
  }
}

// S2: resetShip (game.cpp:133-149): rejection-sample an integer spawn inside the big and outside the small
// hexagon, then the heading. Out of line (rare); takes and returns plain values so the caller's env stays in
// registers. Returns {x, y, angle, new ring index}; *calls = number of rand() calls consumed.
__device__ __noinline__ int4 sf_spawn_draw(unsigned* rng, int np, int i, const SfHot* T, int idx, int* calls) {
  int x, y, n = 0;
  for (;;) {
    x = sf_rand_raw(rng, np, i, idx) % 380 + 170;
    y = sf_rand_raw(rng, np, i, idx) % 330 + 150;
    n += 2;
    if (sf_inside_hex(T, 0, (double)x, (double)y) && !sf_inside_hex(T, 1, (double)x, (double)y)) break;
  }
  int ang = sf_rand_raw(rng, np, i, idx) % 360;
  *calls = n + 1;
  return make_int4(x, y, ang, idx);
}
__device__ __forceinline__ void sf_spawn_ship(const SfDev& D, const SfHot* H, int i, SfEnv& e) {
  int calls = 0;
  int4 sp = sf_spawn_draw(D.rng, D.n_pad, i, H, e.st3.y, &calls);
  e.st3.y = sp.w; e.st3.z += calls;
  e.pos = make_double2((double)sp.x, (double)sp.y);
  e.vel = make_double2(H->ship_start_vx, H->ship_start_vy);
  e.q0.x = (e.q0.x & ~SF_CORE_ANGLE_MASK) | (unsigned)sp.z | SF_CORE_SHIP_ALIVE;
}

// S1: Game::Game (game.cpp:18-82) through SSF_Env.reset (ssf_env.py:163-178). prev_vlner (q1.w),
// the rand stream (st3.yzw) survive; everything else is a fresh Game.
__device__ inline void sf_new_game(const SfDev& D, const SfHot* H, int i, SfEnv& e) {
  e.q0 = make_int4(0, 0, 0, 0);
  sf_spawn_ship(D, H, i, e);
  e.q0.x |= SF_CORE_FORT_ALIVE | (18u << SF_CORE_FANG_SHIFT);  // mAngle=180, mLastAngle=0 (game.cpp:40-41)
  e.q1 = make_int4(0, 250, 0, e.q1.w);                           // mVulnerabilityTimer: 0 + 250 (game.cpp:78)
  e.q2 = make_int4(0, 0, 0, 0);
  e.q3 = make_int4(0, 0, 0, 0);
  D.st0[i] = make_int4(0, 0, 0, 0); D.st1[i] = make_int4(0, 0, 0, 0); D.st2[i] = make_int4(0, 0, 0, 0);  // the Stats of a fresh Game
  e.d0 = 0u; e.d1 = 0u; e.d2 = 0u;
  e.st3.x = 0;
}

// first dead slot (game.cpp:160-172,177-190)
__device__ __forceinline__ int sf_first_free(unsigned mask, int n) {
  unsigned freebits = ~mask & ((1u << n) - 1u);
  return freebits ? __ffs(freebits) - 1 : -1;
}

// One SSF_Env.step: keymask -> key events -> stepOneTick(34) -> shaping -> done -> auto-reset.
__device__ inline void sf_env_step(const SfDev& D, const SfHot* T, int i, SfEnv& e, int keymask, bool autoreset, bool raw_reward, SfStepOut& out) {
  const int np = D.n_pad;
  SF_ST_BEGIN(__activemask());  // the lanes that step an env
  float rew = 0.f;
  unsigned ev = 0;
  unsigned core = (unsigned)e.q0.x;
  if (D.autoturn) keymask &= (SF_KEY_FIRE | SF_KEY_THRUST);  // autoturn envs send only FIRE, THRUST (ssf_env.py:213-220)

  // ---- S3/S4 processKeyState (game.cpp:218-272), events in the order FIRE, THRUST, LEFT, RIGHT ----
  {
    bool pressed = keymask & SF_KEY_FIRE, flag = core & SF_CORE_FIRE;
    if (pressed && !flag) {
      // S5 fireMissile with the PRE-move pose (quirk Q2); totalShots counts even without a missile (Q6)
      if (core & SF_CORE_SHIP_ALIVE) {
        int slot = sf_first_free((unsigned)e.q0.y & SF_PMASK_MISSILES, SF_MAX_MISSILES);
        if (slot >= 0) {
          e.q0.y |= 1 << slot;
          D.mpos[(size_t)slot * np + i] = e.pos;
          D.mang[(size_t)slot * np + i] = (short)(core & SF_CORE_ANGLE_MASK);
          ev |= SF_EV_MISSILE_FIRED;
          sf_reward(e, rew, -D.missile_penalty);
        }
      }
      core |= SF_CORE_FIRE; e.q2.x = 0; SF_ST_INC(e.d1, 3); ev |= SF_EV_PRESS_FIRE;
    } else if (!pressed && flag) { core &= ~SF_CORE_FIRE; e.q2.x = 0; }
    pressed = keymask & SF_KEY_THRUST; flag = core & SF_CORE_THRUST;
    if (pressed && !flag) { core |= SF_CORE_THRUST; e.q2.y = 0; SF_ST_INC(e.d2, 0); ev |= SF_EV_PRESS_THRUST; }
    else if (!pressed && flag) { core &= ~SF_CORE_THRUST; e.q2.y = 0; }
    if (!D.autoturn) {
      pressed = keymask & SF_KEY_LEFT; flag = core & SF_CORE_LEFT;
      if (pressed && !flag) { core |= SF_CORE_LEFT; e.q2.z = 0; SF_ST_INC(e.d2, 1); ev |= SF_EV_PRESS_LEFT; }
      else if (!pressed && flag) { core &= ~SF_CORE_LEFT; e.q2.z = 0; }
      pressed = keymask & SF_KEY_RIGHT; flag = core & SF_CORE_RIGHT;
      if (pressed && !flag) { core |= SF_CORE_RIGHT; e.q2.w = 0; SF_ST_INC(e.d2, 2); ev |= SF_EV_PRESS_RIGHT; }
      else if (!pressed && flag) { core &= ~SF_CORE_RIGHT; e.q2.w = 0; }
    }
  }
  e.q0.x = (int)core;

  // ---- S6 monitorShipRespawn (game.cpp:151-157) ----
  if (!(core & SF_CORE_SHIP_ALIVE) && e.q0.z >= 1000) {
    sf_spawn_ship(D, T, i, e);
    e.q0.w = 0;
    ev |= SF_EV_SHIP_RESPAWN;
    core = (unsigned)e.q0.x;
  }

  SF_ST(9);
  // ---- S7 updateShip (game.cpp:314-351) ----
  if (core & SF_CORE_SHIP_ALIVE) {
    int ang = core & SF_CORE_ANGLE_MASK;
    if (D.autoturn) {
      ang = sf_ceil_angle<1>(T, SF_DSUB(SF_FORT_Y, e.pos.y), SF_DSUB(SF_FORT_X, e.pos.x), true);  // ceil(angleTo), pre-move (Q3)
      if (ang >= 360) ang -= 360;  // stdAngle
    } else {
      bool l = core & SF_CORE_LEFT, r = core & SF_CORE_RIGHT;
      if (l && !r) { ang -= 6; if (ang < 0) ang += 360; }
      else if (r && !l) { ang += 6; if (ang >= 360) ang -= 360; }
    }
    core = (core & ~SF_CORE_ANGLE_MASK) | (unsigned)ang;
    if (core & SF_CORE_THRUST) {
      e.vel.x = SF_DADD(e.vel.x, SF_DMUL(0.3, T->cs[ang][0]));
      e.vel.y = SF_DADD(e.vel.y, SF_DMUL(0.3, T->cs[ang][1]));
    }
    e.pos.x = SF_DADD(e.pos.x, e.vel.x);
    e.pos.y = SF_DADD(e.pos.y, e.vel.y);
    e.q0.x = (int)core;
    if (!sf_inside_hex(T, 0, e.pos.x, e.pos.y)) {
      sf_kill_ship(e); sf_reward(e, rew, -(float)D.death_penalty); SF_ST_INC(e.d0, 0);
      ev |= SF_EV_EXPLODE_BIGHEX | SF_EV_COL_BIGHEX;
    } else if (sf_inside_hex(T, 1, e.pos.x, e.pos.y)) {
      sf_kill_ship(e); sf_reward(e, rew, -(float)D.death_penalty); SF_ST_INC(e.d0, 1);
      ev |= SF_EV_EXPLODE_SMALLHEX | SF_EV_COL_SMALLHEX;
    }
    core = (unsigned)e.q0.x;
  }

  SF_ST(10);
  // ---- S11 updateFortress (game.cpp:194-216) ----
  {
    if (!(core & SF_CORE_FORT_ALIVE) && e.q1.x > 1000) {
      e.q0.w = 0; core |= SF_CORE_FORT_ALIVE; ev |= SF_EV_FORTRESS_RESPAWN;
    }
    if (core & SF_CORE_SHIP_ALIVE) {  // the fortress only tracks a live ship
      const double fdy = SF_DSUB(e.pos.y, SF_FORT_Y), fdx = SF_DSUB(e.pos.x, SF_FORT_X);
      int sect = sf_ceil_angle<10>(T, fdy, fdx, false) / 10;  // ceil(angle_to_ship / 10)
      if (sect >= 36) sect -= 36;
      unsigned last = (core >> SF_CORE_FLAST_SHIFT) & 63u;
      core = (core & ~(63u << SF_CORE_FANG_SHIFT)) | ((unsigned)sect << SF_CORE_FANG_SHIFT);
      if ((unsigned)sect != last) {
        core = (core & ~(63u << SF_CORE_FLAST_SHIFT)) | ((unsigned)sect << SF_CORE_FLAST_SHIFT);
        e.q0.w = 0;
      }
      if (e.q0.w >= 1000 && (core & SF_CORE_FORT_ALIVE)) {
        // S12 fireShell with the exact (real) angle: stdAngle(rad2deg(atan2(dy, dx))) (game.cpp:197), needed here only
        int slot = sf_first_free(((unsigned)e.q0.y >> SF_PMASK_SHELL_SHIFT) & 0xFu, SF_DEV_SHELLS);
        if (slot >= 0) {
          double a = sf_rad2deg(sf_atan2(T, fdy, fdx));
          if (a < 0) a = SF_DADD(a, 360.0);  // stdAngle on (-180,180]
          e.q0.y |= 1 << (SF_PMASK_SHELL_SHIFT + slot);
          D.spos[(size_t)slot * np + i] = make_double2(SF_FORT_X, SF_FORT_Y);
          D.svel[(size_t)slot * np + i] = sf_shell_velocity(a);
          D.sang[(size_t)slot * np + i] = a;
          ev |= SF_EV_FORTRESS_FIRED;
        }
        e.q0.w = 0;
      }
    }
    e.q0.x = (int)core;
  }

  SF_ST(11);
  // ---- S13 updateShells (game.cpp:404-423), slot order ----
  const double thr_ship = T->touch2[0], thr_fort = T->touch2[1], thr_hide = T->touch2[2];
  unsigned vis = 0;
  for (unsigned m = ((unsigned)e.q0.y >> SF_PMASK_SHELL_SHIFT) & 0xFu; m; m &= m - 1) {
    int s = __ffs(m) - 1;
    double2 p = D.spos[(size_t)s * np + i], v = D.svel[(size_t)s * np + i];
    p.x = SF_DADD(p.x, v.x); p.y = SF_DADD(p.y, v.y);
    D.spos[(size_t)s * np + i] = p;
    if ((e.q0.x & SF_CORE_SHIP_ALIVE) && sf_dist2(p.x, p.y, e.pos.x, e.pos.y) <= thr_ship) {
      e.q0.y &= ~(1 << (SF_PMASK_SHELL_SHIFT + s));
      sf_kill_ship(e); sf_reward(e, rew, -(float)D.death_penalty); SF_ST_INC(e.d0, 2);
      ev |= SF_EV_SHELL_HIT_SHIP | SF_EV_COL_SHELL_SHIP;
    } else if (sf_outside(p.x, p.y)) {
      e.q0.y &= ~(1 << (SF_PMASK_SHELL_SHIFT + s));
    } else if (sf_dist2(p.x, p.y, SF_FORT_X, SF_FORT_Y) > thr_hide) vis |= 1u << s;  // quirk Q9: drawn only when further than 21
  }
  out.shell_vis = vis;

  SF_ST(12);
  // ---- S14 updateMissiles (game.cpp:353-402), slot order (order dependent) ----
  for (unsigned m = (unsigned)e.q0.y & SF_PMASK_MISSILES; m; m &= m - 1) {
    int s = __ffs(m) - 1;
    double2 p = D.mpos[(size_t)s * np + i];
    int ang = D.mang[(size_t)s * np + i];
    p.x = SF_DADD(p.x, SF_DMUL(20.0, T->cs[ang][0]));
    p.y = SF_DADD(p.y, SF_DMUL(20.0, T->cs[ang][1]));
    D.mpos[(size_t)s * np + i] = p;
    if (sf_dist2(p.x, p.y, SF_FORT_X, SF_FORT_Y) <= thr_fort) {
      e.q0.y &= ~(1 << s);
      ev |= SF_EV_COL_MISSILE_FORTRESS;
      if (e.q0.x & SF_CORE_FORT_ALIVE) {
        ev |= SF_EV_HIT_FORTRESS;
        if (e.q1.y >= 250) {
          e.q1.z += 1; ev |= SF_EV_VLNER_INCREASED; SF_ST_INC(e.d2, 3);
          if (e.q1.z > e.st3.x) e.st3.x = e.q1.z;
        } else {
          if (e.q1.z >= 11) {
            e.q0.x &= ~SF_CORE_FORT_ALIVE; e.q1.x = 0;
            sf_reward(e, rew, (float)D.destroy_fortress);
            ev |= SF_EV_FORTRESS_DESTROYED; SF_ST_INC(e.d1, 1);
          } else { ev |= SF_EV_VLNER_RESET; SF_ST_INC(e.d1, 0); }
          e.q1.z = 0;
        }
        e.q1.y = 0;
      } else ev |= SF_EV_HIT_DEAD_FORTRESS;
    } else if (sf_outside(p.x, p.y)) {
      e.q0.y &= ~(1 << s);
      sf_reward(e, rew, -0.0f);  // missPenalty == 0 (configs.cpp:11)
      SF_ST_INC(e.d1, 2); ev |= SF_EV_MISSED_SHOT;
    }
  }

  SF_ST(13);
  // ---- S16 stepTimers (game.cpp:425-451) ----
  core = (unsigned)e.q0.x;
  e.q3.z += 1;
  e.q0.w += SF_TICK_MS; e.q1.x += SF_TICK_MS; e.q1.y += SF_TICK_MS; e.q0.z += SF_TICK_MS;
  e.q2.x += (core & SF_CORE_FIRE) ? 1 : -1;
  e.q2.y += (core & SF_CORE_THRUST) ? 1 : -1;
  e.q2.z += (core & SF_CORE_LEFT) ? 1 : -1;
  e.q2.w += (core & SF_CORE_RIGHT) ? 1 : -1;

  // ---- S17 `int stepOneTick`: float -> int truncation (Q1) ; P3 shaping (ssf_env.py:233-244) ----
  int reward = __float2int_rz(rew);
  bool fort_kill = reward > 0;
  if (D.shaped && !raw_reward) {
    int vl = e.q1.z, change = vl - e.q1.w;
    if (vl <= 10 && !fort_kill) reward += change;
    reward = max(-1, min(1, reward));
    reward += fort_kill ? 2 : 0;
    e.q1.w = vl;
  }
  e.q3.w += reward;
  bool done = e.q3.z * SF_TICK_MS >= SF_GAME_TIME;  // isGameOver (game.cpp:487-489)
  out.reward = reward; out.fort_kill = fort_kill; out.done = done;
  if (done && autoreset) ev |= SF_EV_EPISODE_RESET;
  out.events = ev;
  SF_ST(14);
}
