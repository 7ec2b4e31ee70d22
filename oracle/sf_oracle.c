/* TEST INFRASTRUCTURE ONLY (oracle/) — see sf_oracle.h for the parity status.
 *
 * Plain-C restatement of the reference's per-tick game logic, written from
 * the behaviour documented in SURVEY.md §8(a) and checked line by line
 * against the reference (citations are into
 * /root/reference/python/spacefortress/src unless stated otherwise).
 * All state lives in one flat sfr_record; there is no Config map, no event
 * strings and no heap allocation. */
#define _GNU_SOURCE
#include "sf_oracle.h"

#include <math.h>
#include <stdio.h>
#include <string.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* ---- constants actually read on the hot path (configs.cpp:3-89) ---- */
#define TICK_MS 34               /* ssf_env.py:61 */
#define GAME_TIME 180000         /* configs.cpp:55,66,78,86 */
#define AREA_W 710               /* configs.cpp:4 */
#define AREA_H 626               /* configs.cpp:5 */
#define FORT_X 355.0             /* game.cpp:38 */
#define FORT_Y 315.0             /* game.cpp:39 */
#define R_SHIP 10                /* configs.cpp:46 */
#define R_FORT 18                /* configs.cpp:32 */
#define R_MISSILE 5              /* configs.cpp:22 */
#define R_SHELL 3                /* configs.cpp:19 */
#define V_MISSILE 20             /* configs.cpp:21 */
#define V_SHELL 6                /* configs.cpp:18 */
#define SHIP_ACCEL 0.3           /* configs.cpp:47 */
#define SHIP_TURN 6              /* configs.cpp:48 */
#define SECTOR 10                /* configs.cpp:28 */
#define LOCK_TIME 1000           /* configs.cpp:29 */
#define VULN_TIME 250            /* configs.cpp:30 */
#define VULN_THRESHOLD 10        /* configs.cpp:31 */
#define EXPLODE_MS 1000          /* configs.cpp:40 */

typedef struct { int destroy_fortress, death_penalty; double missile_penalty; int autoturn, shaped; } preset;

static preset preset_of(int gametype) {
  preset p;
  /* train presets scale everything to +-1 (configs.cpp:51-72); test presets keep baseConfig's
   * 100 / 100 / 2.0 (configs.cpp:8-10,74-89) */
  int test = (gametype == SFO_TEST_YOUTURN || gametype == SFO_TEST_AUTOTURN);
  p.destroy_fortress = test ? 100 : 1;
  p.death_penalty = test ? 100 : 1;
  p.missile_penalty = test ? 2.0 : 0.05;
  p.autoturn = (gametype == SFO_AUTOTURN || gametype == SFO_TEST_AUTOTURN);
  p.shaped = !test; /* ssf_env.py:235 */
  return p;
}

int sfo_gametype_from_name(const char* name) {
  if (!strcmp(name, "youturn")) return SFO_YOUTURN;
  if (!strcmp(name, "autoturn")) return SFO_AUTOTURN;
  if (!strcmp(name, "test-youturn")) return SFO_TEST_YOUTURN;
  if (!strcmp(name, "test-autoturn")) return SFO_TEST_AUTOTURN;
  return -1;
}

/* ---- G1: glibc rand()/srand(), TYPE_3 additive feedback generator -------
 * (glibc stdlib/random_r.c, published algorithm; call sites game.cpp:137-148).
 * r[0]=seed, r[i]=16807*r[i-1] mod (2^31-1) for i<31 (Schrage form), then the
 * lag-(31,3) sum over uint32, first 310 outputs dropped, output = r>>1. */
void sfo_srand(sfo_env* e, uint32_t seed) {
  if (seed == 0) seed = 1;
  int32_t w = (int32_t)seed;
  e->r[0] = w;
  for (int i = 1; i < 31; i++) {
    long hi = w / 127773, lo = w % 127773;
    long v = 16807 * lo - 2836 * hi;
    if (v < 0) v += 2147483647;
    w = (int32_t)v;
    e->r[i] = w;
  }
  e->rng_i = 34; /* r[31..33] alias r[0..2] in a 31-word ring */
  e->s.rng_seed = seed;
  for (int k = 0; k < 310; k++) (void)sfo_rand(e);
  e->s.rng_count = 0;
}

int sfo_rand(sfo_env* e) {
  int i = e->rng_i;
  uint32_t v = (uint32_t)e->r[i % 31] + (uint32_t)e->r[(i - 3) % 31];
  e->r[i % 31] = (int32_t)v;
  e->rng_i = (i + 1 == 34 + 31) ? 34 : i + 1; /* only i mod 31 matters */
  e->s.rng_count++;
  return (int)(v >> 1);
}

/* ---- geometry helpers (vector.cpp:34-52, object.cpp:12-15, hexagon.cpp:13-48) ---- */
static double deg2rad(double a) { return a * M_PI / 180; }
static double rad2deg(double a) { return a / M_PI * 180; }
static double std_angle(double a) {
  if (a <= -360 || a >= 360) a = fmod(a, 360);
  if (a < 0) a += 360;
  return a;
}

static void hex_points(int radius, double* px, double* py) {
  /* hexagon.cpp:13-35: vertices are floored to integers */
  double x1 = floor(355 - radius), x2 = floor(355 - radius * 0.5);
  double x3 = floor(355 + radius * 0.5), x4 = floor(355 + radius);
  double y1 = 315, y2 = floor(315 - radius * sin(M_PI * 2 / 3)), y3 = floor(315 + radius * sin(M_PI * 2 / 3));
  px[0] = x1; py[0] = y1; px[1] = x2; py[1] = y2; px[2] = x3; py[2] = y2;
  px[3] = x4; py[3] = y1; px[4] = x3; py[4] = y3; px[5] = x2; py[5] = y3;
}

static int inside_hex(int radius, double x, double y) {
  /* hexagon.cpp:37-48: boundary inclusive */
  double px[6], py[6];
  hex_points(radius, px, py);
  for (int i = 0; i < 6; i++) {
    int j = (i + 1) % 6;
    double nx = -(py[j] - py[i]), ny = px[j] - px[i];
    double dx = x - px[i], dy = y - py[i];
    if (nx * dx + ny * dy < 0) return 0;
  }
  return 1;
}

static int circles_touch(double ax, double ay, double bx, double by, int rsum) {
  /* object.cpp:12-15; pow(x,2) == x*x exactly */
  double dx = ax - bx, dy = ay - by;
  return sqrt(dx * dx + dy * dy) <= rsum;
}

static int outside_area(double x, double y) { /* game.cpp:129-131 */
  return x < 0 || x > AREA_W || y > AREA_H || y < 0;
}

/* ---- S15: reward/penalize in float32 (game.cpp:97-106) ---- */
typedef struct { float reward; } tick_ctx;
static void add_reward(sfo_env* e, tick_ctx* t, float amt) {
  t->reward += amt;
  e->s.raw_points += amt;
  e->s.points += amt;
  if (e->s.points < 0) e->s.points = 0;
}

/* ---- S2: resetShip (game.cpp:133-149) ---- */
static void spawn_ship(sfo_env* e) {
  sfr_record* s = &e->s;
  s->ship_alive = 1;
  for (;;) {
    s->ship_x = sfo_rand(e) % 380 + 170;
    s->ship_y = sfo_rand(e) % 330 + 150;
    if (inside_hex(200, s->ship_x, s->ship_y) && !inside_hex(40, s->ship_x, s->ship_y)) break;
  }
  s->ship_vx = cos(deg2rad(-60)); /* configs.cpp:43-44 */
  s->ship_vy = sin(deg2rad(-60));
  s->ship_angle = sfo_rand(e) % 360;
}

/* ---- S1: Game::Game (game.cpp:18-82) via SSF_Env.reset (ssf_env.py:163-178) ---- */
void sfo_reset(sfo_env* e) {
  sfr_record keep = e->s;
  memset(&e->s, 0, sizeof(e->s));
  e->s.prev_vlner = keep.prev_vlner; /* quirk Q7: survives reset() (ssf_env.py:92) */
  e->s.rng_seed = keep.rng_seed;
  e->s.rng_count = keep.rng_count;
  spawn_ship(e);
  e->s.fortress_alive = 1;
  e->s.fortress_angle = 180;  /* game.cpp:40 */
  e->s.fortress_last_angle = 0;
  e->s.fortress_vuln_timer = VULN_TIME; /* game.cpp:78 on a zeroed member (quirk Q5) */
}

void sfo_create(sfo_env* e, int gametype, uint32_t seed) {
  memset(e, 0, sizeof(*e));
  e->gametype = gametype;
  sfo_srand(e, seed);
  e->s.prev_vlner = 0;
  sfo_reset(e);
}

void sfo_set_state(sfo_env* e, const sfr_record* r) {
  uint32_t n = r->rng_count;
  sfo_srand(e, r->rng_seed);
  for (uint32_t i = 0; i < n; i++) (void)sfo_rand(e);
  e->s = *r;
  e->s.rng_count = n;
}

/* ---- S5 / S12: first dead slot of 20 (game.cpp:159-192) ---- */
static int first_free(uint32_t mask, int n) {
  for (int i = 0; i < n; i++) if (!((mask >> i) & 1)) return i;
  return -1;
}

static void fire_missile(sfo_env* e, tick_ctx* t, const preset* p, uint32_t* ev) {
  sfr_record* s = &e->s;
  if (!s->ship_alive) return;
  int i = first_free(s->missile_mask, SFR_MAX_MISSILES);
  if (i < 0) return; /* no slot: no missile and no penalty */
  s->missile_mask |= 1u << i;
  s->missile_x[i] = s->ship_x; s->missile_y[i] = s->ship_y; /* pre-move pose, quirk Q2 */
  s->missile_angle[i] = s->ship_angle;
  s->missile_vx[i] = V_MISSILE * cos(deg2rad(s->ship_angle));
  s->missile_vy[i] = V_MISSILE * sin(deg2rad(s->ship_angle));
  *ev |= SFE_MISSILE_FIRED;
  add_reward(e, t, -(float)p->missile_penalty);
}

static void fire_shell(sfo_env* e, double angle, uint32_t* ev) {
  sfr_record* s = &e->s;
  int i = first_free(s->shell_mask, SFR_MAX_SHELLS);
  if (i < 0) return;
  s->shell_mask |= 1u << i;
  s->shell_x[i] = FORT_X; s->shell_y[i] = FORT_Y;
  s->shell_angle[i] = angle;
  s->shell_vx[i] = V_SHELL * cos(deg2rad(angle));
  s->shell_vy[i] = V_SHELL * sin(deg2rad(angle));
  *ev |= SFE_FORTRESS_FIRED;
}

/* ---- S10: killShip (game.cpp:274-280) ---- */
static void kill_ship(sfr_record* s) {
  if (s->ship_alive) { s->ship_alive = 0; s->ship_death_timer = 0; s->stats[3]++; }
}

/* ---- S3/S4: key events in the order the env sends them (ssf_env.py:213-229),
 * processed as in game.cpp:218-272 ---- */
static void one_key(sfo_env* e, tick_ctx* t, const preset* p, int bit, int pressed, uint32_t* ev) {
  sfr_record* s = &e->s;
  int32_t *flag, *timer;
  switch (bit) {
    case SFK_FIRE: flag = &s->fire_flag; timer = &s->fire_timer; break;
    case SFK_THRUST: flag = &s->thrust_flag; timer = &s->thrust_timer; break;
    case SFK_LEFT: flag = &s->left_flag; timer = &s->left_timer; break;
    default: flag = &s->right_flag; timer = &s->right_timer; break;
  }
  if (pressed && !*flag) {
    if (bit == SFK_FIRE) { fire_missile(e, t, p, ev); s->stats[7]++; *ev |= SFE_PRESS_FIRE; } /* totalShots even with no slot / dead ship (Q6) */
    else if (bit == SFK_THRUST) { s->stats[8]++; *ev |= SFE_PRESS_THRUST; }
    else if (bit == SFK_LEFT) { s->stats[9]++; *ev |= SFE_PRESS_LEFT; }
    else { s->stats[10]++; *ev |= SFE_PRESS_RIGHT; }
    *flag = 1; *timer = 0;
  } else if (!pressed && *flag) {
    *flag = 0; *timer = 0; /* the duration vectors (S20) are not kept */
  }
}

/* ---- S17: Game::stepOneTick (game.cpp:473-485) ---- */
int sfo_core_step(sfo_env* e, int keymask, uint32_t* events) {
  sfr_record* s = &e->s;
  preset p = preset_of(e->gametype);
  tick_ctx t; t.reward = 0;
  uint32_t ev = 0;
  int youturn = !p.autoturn;

  s->time += TICK_MS; /* updateTime */

  /* processKeyState */
  one_key(e, &t, &p, SFK_FIRE, keymask & SFK_FIRE, &ev);
  one_key(e, &t, &p, SFK_THRUST, keymask & SFK_THRUST, &ev);
  if (youturn) {
    one_key(e, &t, &p, SFK_LEFT, keymask & SFK_LEFT, &ev);
    one_key(e, &t, &p, SFK_RIGHT, keymask & SFK_RIGHT, &ev);
  }
  s->turn_flag = (s->left_flag && !s->right_flag) ? 1 : (!s->left_flag && s->right_flag) ? 2 : 0;

  /* S6 monitorShipRespawn (game.cpp:151-157) */
  if (!s->ship_alive && s->ship_death_timer >= EXPLODE_MS) {
    spawn_ship(e);
    s->fortress_timer = 0;
    ev |= SFE_SHIP_RESPAWN;
  }

  /* S7 updateShip (game.cpp:314-351) */
  if (s->ship_alive) {
    if (p.autoturn) {
      double a = atan2(FORT_Y - s->ship_y, FORT_X - s->ship_x); /* angleTo, vector.cpp:48-52 */
      if (a < 0) a += M_PI * 2;
      s->ship_angle = std_angle(ceil(rad2deg(a)));
    } else if (s->turn_flag == 1) {
      s->ship_angle = std_angle(s->ship_angle - SHIP_TURN);
    } else if (s->turn_flag == 2) {
      s->ship_angle = std_angle(s->ship_angle + SHIP_TURN);
    }
    if (s->thrust_flag) {
      s->ship_vx += SHIP_ACCEL * cos(deg2rad(s->ship_angle));
      s->ship_vy += SHIP_ACCEL * sin(deg2rad(s->ship_angle));
    }
    s->ship_x += s->ship_vx;
    s->ship_y += s->ship_vy;
    if (!inside_hex(200, s->ship_x, s->ship_y)) {
      kill_ship(s);
      add_reward(e, &t, -(float)p.death_penalty);
      s->stats[0]++;
      ev |= SFE_EXPLODE_BIGHEX | SFE_COL_BIGHEX;
    } else if (inside_hex(40, s->ship_x, s->ship_y)) {
      kill_ship(s);
      add_reward(e, &t, -(float)p.death_penalty);
      s->stats[1]++;
      ev |= SFE_EXPLODE_SMALLHEX | SFE_COL_SMALLHEX;
    }
  }

  /* S11 updateFortress (game.cpp:194-216) */
  {
    double ang = std_angle(rad2deg(atan2(s->ship_y - FORT_Y, s->ship_x - FORT_X)));
    if (!s->fortress_alive && s->fortress_death_timer > 1000) {
      s->fortress_timer = 0;
      s->fortress_alive = 1;
      ev |= SFE_FORTRESS_RESPAWN;
    }
    if (s->ship_alive) {
      s->fortress_angle = std_angle(ceil(ang / SECTOR) * SECTOR);
      if (s->fortress_angle != s->fortress_last_angle) {
        s->fortress_last_angle = s->fortress_angle;
        s->fortress_timer = 0;
      }
      if (s->fortress_timer >= LOCK_TIME && s->fortress_alive) {
        fire_shell(e, ang, &ev);
        s->fortress_timer = 0;
      }
    }
  }

  /* S13 updateShells (game.cpp:404-423) */
  for (int i = 0; i < SFR_MAX_SHELLS; i++) {
    if (!((s->shell_mask >> i) & 1)) continue;
    s->shell_x[i] += s->shell_vx[i];
    s->shell_y[i] += s->shell_vy[i];
    if (s->ship_alive && circles_touch(s->shell_x[i], s->shell_y[i], s->ship_x, s->ship_y, R_SHELL + R_SHIP)) {
      s->shell_mask &= ~(1u << i);
      kill_ship(s);
      add_reward(e, &t, -(float)p.death_penalty);
      s->stats[2]++;
      ev |= SFE_SHELL_HIT_SHIP | SFE_COL_SHELL_SHIP;
    } else if (outside_area(s->shell_x[i], s->shell_y[i])) {
      s->shell_mask &= ~(1u << i);
    }
  }

  /* S14 updateMissiles (game.cpp:353-402) */
  for (int i = 0; i < SFR_MAX_MISSILES; i++) {
    if (!((s->missile_mask >> i) & 1)) continue;
    s->missile_x[i] += s->missile_vx[i];
    s->missile_y[i] += s->missile_vy[i];
    if (circles_touch(s->missile_x[i], s->missile_y[i], FORT_X, FORT_Y, R_MISSILE + R_FORT)) {
      s->missile_mask &= ~(1u << i);
      ev |= SFE_COL_MISSILE_FORTRESS;
      if (s->fortress_alive) {
        ev |= SFE_HIT_FORTRESS;
        if (s->fortress_vuln_timer >= VULN_TIME) {
          s->vulnerability++;
          ev |= SFE_VLNER_INCREASED;
          s->stats[11]++;
          if (s->vulnerability > s->stats[12]) s->stats[12] = s->vulnerability;
        } else {
          if (s->vulnerability >= VULN_THRESHOLD + 1) {
            s->fortress_alive = 0;
            s->fortress_death_timer = 0;
            add_reward(e, &t, (float)(p.destroy_fortress + 0)); /* mDestroyFortressExtraPoints == 0 */
            ev |= SFE_FORTRESS_DESTROYED;
            s->stats[5]++;
          } else {
            ev |= SFE_VLNER_RESET;
            s->stats[4]++;
          }
          s->vulnerability = 0;
        }
        s->fortress_vuln_timer = 0;
      } else {
        ev |= SFE_HIT_DEAD_FORTRESS;
      }
    } else if (outside_area(s->missile_x[i], s->missile_y[i])) {
      s->missile_mask &= ~(1u << i);
      add_reward(e, &t, -0.0f); /* missPenalty == 0 (configs.cpp:11) */
      s->stats[6]++;
      ev |= SFE_MISSED_SHOT;
    }
  }

  /* S16 stepTimers (game.cpp:425-451): death timers tick even while alive (Q4) */
  s->tick += 1;
  s->fortress_timer += TICK_MS;
  s->fortress_death_timer += TICK_MS;
  s->fortress_vuln_timer += TICK_MS;
  s->ship_death_timer += TICK_MS;
  s->fire_timer += s->fire_flag ? 1 : -1;
  s->thrust_timer += s->thrust_flag ? 1 : -1;
  s->left_timer += s->left_flag ? 1 : -1;
  s->right_timer += s->right_flag ? 1 : -1;

  if (events) *events = ev;
  return (int)t.reward; /* `int stepOneTick` returns the float: truncation (Q1), pymodule.cpp:230 */
}

/* ---- P3-P5: SSF_Env.step shaping (ssf_env.py:231-250) ---- */
void sfo_env_step(sfo_env* e, int keymask, int* out4) {
  uint32_t ev = 0;
  int reward = sfo_core_step(e, keymask, &ev);
  int fort_kill = reward > 0;
  preset p = preset_of(e->gametype);
  if (p.shaped) {
    int vl = e->s.vulnerability;
    int change = vl - e->s.prev_vlner;
    if (vl <= 10 && !fort_kill) reward += change;
    if (reward > 1) reward = 1;
    if (reward < -1) reward = -1;
    reward += 2 * fort_kill;
    e->s.prev_vlner = vl;
  }
  out4[0] = reward;
  out4[1] = e->s.time >= GAME_TIME; /* isGameOver, game.cpp:487-489 */
  out4[2] = fort_kill;
  out4[3] = (int)ev;
}

/* teacher-forced single steps over an array of states: recs[i] <- the state after sfo_env_step(keymask) from recs[i]
 * (a fresh env of the game type each, the rand stream re-derived from the record); out4[4 * i ..] as sfo_env_step */
void sfo_step_records(int gametype, sfr_record* recs, long n, int keymask, int* out4) {
  sfo_env e;
  for (long i = 0; i < n; i++) {
    memset(&e, 0, sizeof(e));
    e.gametype = gametype;
    sfo_set_state(&e, &recs[i]);
    sfo_env_step(&e, keymask, out4 + 4 * i);
    recs[i] = e.s;
  }
}

/* ---- P2: action tables (ssf_env.py:65-90) ---- */
int sfo_num_actions(int gametype, int action_set) {
  int youturn = (gametype == SFO_YOUTURN || gametype == SFO_TEST_YOUTURN);
  if (action_set == 1) return youturn ? 5 : 3;
  if (action_set == -1) return 16;
  if (action_set == 0) return youturn ? 16 : 4;
  return -1;
}

int sfo_action_to_keymask(int gametype, int action_set, int action) {
  int youturn = (gametype == SFO_YOUTURN || gametype == SFO_TEST_YOUTURN);
  int n = sfo_num_actions(gametype, action_set);
  if (n < 0 || action < 0 || action >= n) return -1;
  if (action_set == 1) {
    static const int tab[5] = {0, SFK_FIRE, SFK_THRUST, SFK_LEFT, SFK_RIGHT};
    return tab[action];
  }
  /* np.array(np.meshgrid(a0,a1[,a2,a3])).T.reshape(-1,k): with numpy's default 'xy'
   * indexing the row r of the result has column c given by the digit table below
   * (verified against numpy in tests/test_actions.py). */
  if (n == 4) { /* meshgrid([0,1],[0,1]).T.reshape(-1,2): rows (0,0),(0,1),(1,0),(1,1) */
    int fire = (action >> 1) & 1, thrust = action & 1;
    int m = (fire ? SFK_FIRE : 0) | (thrust ? SFK_THRUST : 0);
    return m;
  }
  /* 4-D case: row index r = ((i3*2 + i2)*2 + i0)*2 + i1 where ik indexes input k;
   * columns are (a0,a1,a2,a3) = (fire,thrust,left,right) */
  {
    int i1 = action & 1, i0 = (action >> 1) & 1, i2 = (action >> 2) & 1, i3 = (action >> 3) & 1;
    int m = (i0 ? SFK_FIRE : 0) | (i1 ? SFK_THRUST : 0) | (i2 ? SFK_LEFT : 0) | (i3 ? SFK_RIGHT : 0);
    if (!youturn) m &= (SFK_FIRE | SFK_THRUST); /* autoturn only reads keystate[0:2] (ssf_env.py:213-220) */
    return m;
  }
}

/* ---- S8: computeExtra (game.cpp:282-312), evaluated on demand from the
 * (frozen-while-dead) ship state; includes the fdist bug (Q11) ---- */
void sfo_get_extra(const sfo_env* e, double* out4) {
  const sfr_record* s = &e->s;
  double vdir;
  if (s->tick == 0) { /* no updateShip yet: mExtra of a fresh Game (zero-filled in oracle/ref_harness.cpp) */
    out4[0] = out4[1] = out4[2] = out4[3] = 0.0;
    return;
  }
  if (sqrt(s->ship_vx * s->ship_vx + s->ship_vy * s->ship_vy) == 0.0) vdir = 0.0;
  else {
    double o = atan2(-(FORT_Y - s->ship_y), FORT_X - s->ship_x);
    double v = atan2(s->ship_vy, s->ship_vx);
    double d = v - o;
    if (d > M_PI) d -= M_PI * 2;
    if (d < -M_PI) d += M_PI * 2;
    vdir = rad2deg(d);
  }
  double o = atan2(s->ship_y - FORT_Y, s->ship_x - FORT_X);
  o = rad2deg(o) - s->ship_angle + 180;
  if (o < -180) o = o + 360;
  double dx = s->ship_x - FORT_X, dy0 = s->ship_y - s->ship_y;
  double fdist = sqrt(dx * dx + dy0 * dy0);
  double ndist = -1 + (fdist - 40.0) / ((200.0 - 40.0) / 2.0);
  out4[0] = vdir; out4[1] = fdist; out4[2] = ndist; out4[3] = o;
}

/* ---- Game::dumpState (game.cpp:519-576). The event list is rebuilt from the
 * key mask (press-/release- are logged for every key every tick, game.cpp:223)
 * and the event bits; events that can repeat within a tick (missile hits)
 * appear once, so this string equals the reference's only when no event
 * repeats — the tests use it that way. ---- */
int sfo_dump(const sfo_env* e, int keymask, uint32_t ev, char* buf, int cap) {
  const sfr_record* s = &e->s;
  int n = 0;
#define APP(...) do { n += snprintf(buf + n, n < cap ? (size_t)(cap - n) : 0, __VA_ARGS__); } while (0)
  APP("[%d,%d,%.3f,%.3f,%.3f,%.3f,%.1f,%d,%.1f,[", s->time, s->ship_alive ? 1 : 0, s->ship_x, s->ship_y,
      s->ship_vx, s->ship_vy, s->ship_angle, s->fortress_alive ? 1 : 0, s->fortress_angle);
  int first = 1;
  for (int i = 0; i < SFR_MAX_MISSILES; i++) if ((s->missile_mask >> i) & 1) {
    APP("%s%.3f,%.3f,%.1f", first ? "" : ",", s->missile_x[i], s->missile_y[i], s->missile_angle[i]); first = 0;
  }
  APP("],[");
  first = 1;
  for (int i = 0; i < SFR_MAX_SHELLS; i++) if ((s->shell_mask >> i) & 1) {
    APP("%s%.3f,%.3f,%.1f", first ? "" : ",", s->shell_x[i], s->shell_y[i], s->shell_angle[i]); first = 0;
  }
  APP("],%.1f,%d,%d,%d,[", (double)s->points, s->vulnerability, s->thrust_flag ? 1 : 0, s->turn_flag);
  (void)keymask; (void)ev;
  APP("]]");
#undef APP
  return n;
}

/* bulk run for timing (bench.py cpu_baseline kind "port"): env step + auto-reset
 * (+ frame when obs84_last != NULL) */
long sfo_run(sfo_env* e, const unsigned char* keymasks, long steps, unsigned char* obs84_last) {
  long acc = 0;
  int out[4];
  for (long i = 0; i < steps; i++) {
    sfo_env_step(e, keymasks[i], out);
    acc += out[0];
    if (out[1]) sfo_reset(e);
    if (obs84_last) { sfo_draw_obs(&e->s, obs84_last); acc += obs84_last[(i * 7) % (84 * 84)]; }
  }
  return acc;
}
