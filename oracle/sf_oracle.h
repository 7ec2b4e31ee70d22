/* TEST INFRASTRUCTURE ONLY (oracle/): plain-C CPU restatement of the reference
 * hot path (game tick + env shaping + auto-reset + frame). Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline/reference legs may use it.
 * Parity status: the game-step part is PINNED against the compiled reference
 * core (oracle/_ref, tests/test_oracle_vs_ref.py) and the known answers of
 * SURVEY.md §8(c). The frame part is a restatement of draw.cpp over a
 * documented model of cairo's image backend; real cairo cannot be built or
 * imported offline, so frame parity against real cairo is UNPINNED (the
 * INTER_AREA resize stage alone is pinned against real cv2). */
#ifndef SF_ORACLE_H
#define SF_ORACLE_H
#include <stdint.h>
#include "sf_record.h"

#ifdef __cplusplus
extern "C" {
#endif

enum { SFO_YOUTURN = 0, SFO_AUTOTURN = 1, SFO_TEST_YOUTURN = 2, SFO_TEST_AUTOTURN = 3 };

typedef struct sfo_env {
  sfr_record s;
  int gametype;
  /* glibc TYPE_3 generator state (restated, see sfo_rand) */
  int32_t r[34];
  int rng_i;
} sfo_env;

int sfo_gametype_from_name(const char* name); /* -1 if unknown (pymodule.cpp:331-343) */
void sfo_srand(sfo_env* e, uint32_t seed);
int sfo_rand(sfo_env* e);
void sfo_create(sfo_env* e, int gametype, uint32_t seed); /* = SSF_Env.__init__: seeds the stream, prev_vlner=0, reset */
void sfo_reset(sfo_env* e);                               /* = SSF_Env.reset(): new Game */
int sfo_core_step(sfo_env* e, int keymask, uint32_t* events); /* = press/release keys + Game::stepOneTick(34) */
void sfo_env_step(sfo_env* e, int keymask, int* out4);    /* = SSF_Env.step: out = reward, done, fort_kill, events */
void sfo_set_state(sfo_env* e, const sfr_record* r);      /* teacher forcing (re-derives the rand stream) */
void sfo_step_records(int gametype, sfr_record* recs, long n, int keymask, int* out4); /* sfo_set_state + sfo_env_step per record */
void sfo_get_extra(const sfo_env* e, double* out4);       /* vdir, fdist, ndist, aim (game.cpp:282-312) */
int sfo_dump(const sfo_env* e, int keymask, uint32_t events, char* buf, int cap); /* Game::dumpState */
long sfo_run(sfo_env* e, const unsigned char* keymasks, long steps, unsigned char* obs84_last);
int sfo_action_to_keymask(int gametype, int action_set, int action); /* ssf_env.py:65-90 */
int sfo_num_actions(int gametype, int action_set);

/* ---- frame restatement (sf_draw_oracle.c) ---- */
#define SFO_NATIVE_W 90
#define SFO_NATIVE_H 92
#define SFO_OBS_W 84
#define SFO_OBS_H 84
void sfo_draw_native(const sfr_record* s, uint8_t* gray /* [92*90] */); /* draw.cpp:256-270 + ssf_env.py:205 */
void sfo_resize_area(const uint8_t* src, int sh, int sw, uint8_t* dst, int dh, int dw); /* cv2.resize INTER_AREA, rl/envs.py:29 */
void sfo_draw_obs(const sfr_record* s, uint8_t* obs84 /* [84*84] */);
void sfo_set_glyph_masks(const uint8_t* alpha /* [10][5*27] */, const uint8_t* slot /* [27] */); /* real-font digits (NULL: 7-segment face) */

#ifdef __cplusplus
}
#endif
#endif
