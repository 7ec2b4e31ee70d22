// sf_render.cuh — block-cooperative rasteriser: the 23 drawing warps of a block draw the frames of a group of <= 32
// envs, two ticks per stage, while warp 0 steps the group's next ticks and prepares the next stage.
// Replaces drawGameStateScaled (draw.cpp:256-270), the RGBA2GRAY conversion (ssf_env.py:205, identity on grey
// input) and cv2.resize(INTER_AREA, 84x84) (rl/envs.py:29).
//
// Draw order and semantics follow draw.cpp:227-269:
//   black, 2 hexagons -> ship wireframe | ship explosion -> fortress wireframe | fortress explosion
//   -> missiles -> shells further than 21 from the fortress -> score digits -> vulnerability bar.
//
// Organisation (one block per SM; see the pipeline at the end of this file):
//  * The default observation (hexagons, "0000000", empty bar; 7056 B) of every env goes out as ONE TMA bulk copy from
//    shared memory; the few 16-byte chunks that the fortress state and a non-empty bar change are patched from
//    pre-resampled tables, and the resampled explosion box of a dead ship is copied from a per-env cache.
//  * Everything that moves (ship, missiles, shells) is a wireframe STROKE of 3-4 stroked segments (quads). The strokes
//    of all envs of the round are pooled. B1: every drawing warp builds the geometry of one batch of <= 8 strokes
//    (fp64 CTM, 24.8 fixed point, edge records with magic reciprocals) and opens one REGION per stroke (bounding box
//    in native pixels + 16-bit coverage cells) in block-wide pools. B3: the scan-conversion passes of all batches are
//    dealt round-robin over all drawing warps: one lane per (stroke, sub-row) computes the exact spans of the
//    stroke's quads (integer edge stepping), makes them disjoint (non-zero winding of equally oriented convex quads
//    == union) and adds the lengths to the cells with shared-memory atomics.
//  * C: for every visible stroke (and every stale quarter of a dead ship's explosion box, and a non-zero score) a
//    WINDOW is composited: the native pixels that the box's output pixels read (INTER_AREA footprint closure, at
//    most 30x32) are initialised from the background and EVERY layer of the env that intersects the window is
//    blended in draw order, clipped to it. The window is resampled with cv2's float arithmetic and its output pixels
//    overwrite the static ones. Windows are independent of each other (overlapping windows recompute the same
//    pixels), so no full-frame tile exists anywhere.
//  * The ship explosion (85 strokes) is identical for the 30 ticks a ship stays dead. On the first dead frame it is
//    scan-converted from per-y-phase span tables (SfExpPhase) with register accumulation, composited once per pixel
//    (phase B2) and kept as a 28x28 native sprite per env; the resampled box is cached per quarter as soon as no
//    wireframe reaches into it, and from then on copied instead of recomputed (memos, not game state).
#pragma once
#include "sf_geom.h"
#include "sf_probe.cuh"
#include "sf_state.cuh"
#include "sf_tables.h"

#define SF_BATCH_QUADS 32
#define SF_MAX_GROUPS 256    // (stroke, 8 sub-rows) work groups of one batch: 8 wireframes x <= 30, or 32 one-quad strokes x <= 8
// A window is the INTER_AREA footprint closure of a box of at most 28x28 native pixels (the explosion sprite):
// +1 column each side (<= 2 taps in x), +2 rows each side (<= 3 taps in y) -> at most 30 x 32. Rows are 32 bytes
// apart; the resampler always reads 2 x 3 taps (missing ones have weight 0), i.e. up to row h+1 and column w.
#define SF_PATCH_STRIDE 32
#define SF_PATCH_BYTES (36 * 32)
#define SF_WIN_MAX_W 31
#define SF_WIN_MAX_H 34
#define SF_YBIAS 4096        // grid rows are stored biased so they fit an unsigned 16-bit field
#define SF_TAG_SHIP 0
#define SF_TAG_PROJECTILE 1
#define SF_SPAN_NONE 0xFFFFFFFFu
#define SF_QF_IRREGULAR 2    // quad flag: not a 2+2 edge split, test all four edges

#define SF_RENDER_WARPS 24   // warps per block (one block per SM): warp 0 steps, the others draw; 80 registers per thread
#define SF_FORT_LIST_SMEM 48                     // lit pixels of a fortress sprite kept in shared memory (the sprites have <= 42)
#define SF_GROUP_ENVS 32                         // envs a block renders per tick: one per lane of the stepping warp
#define SF_STAGE_TICKS 2                         // consecutive ticks of the group drawn together in one stage
#define SF_STAGE_SLOTS (SF_GROUP_ENVS * SF_STAGE_TICKS)  // env slot = 32 * (tick within the stage) + lane of the env
#define SF_ROUND_STROKES (8 * (SF_RENDER_WARPS - 1))  // strokes pooled per round: one batch of <= 8 per drawing warp (a round takes as many envs of the group as fit)
// Block-wide pools of a round: one region (bounding box in native pixels + coverage cells) per visible stroke.
// The round scan admits envs by WORST-CASE need, so the pools cannot overflow: a ship wireframe spans at most
// 44 user units (8.8 px) + the line width in any direction, a missile 25 (5 px), a shell 24 (4.8 px).
#define SF_CELLS_SHIP 144
#define SF_CELLS_MISSILE 49
#define SF_CELLS_SHELL 49
#define SF_POOL_CELLS 12288                      // 16-bit coverage cells
#define SF_POOL_REGIONS SF_ROUND_STROKES
// B1 is latency bound (a batch of 8 strokes takes as long as one of 4), and every batch rounds its last pass of B3 up:
#define SF_CHUNK_WARPS 12  // about 12 batches per round measured best (22: +1 % more passes; 8: the same)


// per-warp shared memory (3.6 KB): the records of the batch being scan-converted; the window being composited
// aliases the edge records (compositing starts after the block's last batch)
struct __align__(16) SfWarpSmem {
  union {
    int4 edge[SF_BATCH_QUADS * 4];          // 2048 B per quad: down A,B, up A,B = {x0, yref | yother<<16 (biased), dx, magic}
    unsigned char patch[SF_PATCH_BYTES];    // 1152 B native pixels of the window
  };
  int4 qinfo[SF_BATCH_QUADS];               //  512 B per quad: {g0 | g1<<16 (biased, clipped to the region), splitD | splitU<<16, flags, 0}
  int4 srec[SF_BATCH_QUADS];                //  512 B per stroke slot: {x0 | w<<8 | nq<<16 | quad0<<24, top (biased), first cell, s0 | s1<<16}
  unsigned short glist[SF_MAX_GROUPS];      //  512 B slot | k<<5 : sub-rows s0 + 8k .. s0 + 8k + 7 of a stroke
  int ngroups, pad0, pad1, pad2;
};

// what the renderer needs to know about one env of the block's group (written by the lane that stepped it)
struct __align__(16) SfEnvRec {
  double px, py;              // ship position (wireframe / explosion centre)
  unsigned core, pmask;       // sf_state.cuh: q0.x, q0.y
  int points_i, vuln, kill_bar;  // (int)mPoints, mVulnerability, vuln > 10 && vulnerability timer < 250 (draw.cpp:268)
  int env;                    // index into the slab; -1: slot unused / masked out
  int s0, ns;                 // this env's strokes in the round's list (draw order)
  int ebox;                   // dead ship: explosion sprite box origin (bx0+64) | (by0+64)<<8
  int shell_vis;              // shells further than 21 from the fortress (quirk Q9), bit per slot
  int building;               // bit 0: dead ship whose explosion sprite is not cached yet: its arcs are scan-converted this round;
                              // bits 4..7: quarters of its resampled explosion box that are valid in D.expo (copied, not recomputed)
  unsigned life;              // rand() calls consumed when this ship spawned + 1: names the explosion of this life
};
// what, besides the explosion itself, lies under a dead ship's explosion box: fortress state | bar state | score
__device__ __forceinline__ unsigned sf_expo_key(const SfEnvRec& r) {
  const int fst = (r.core & (1u << 22)) ? (int)((r.core >> 9) & 63u) : 36;   // SF_CORE_FORT_ALIVE, SF_CORE_FANG_SHIFT
  const int bst = r.kill_bar ? 11 : min(r.vuln, 10);
  return (unsigned)fst | ((unsigned)bst << 6) | (((unsigned)r.points_i & 0x3FFFFu) << 10);
}
// one moving wireframe of the round: desc = kind | angle<<2 | env slot<<12 (its region is in SfStagePool::stroke_region)
struct __align__(8) SfStrokeRec { double x, y; int desc; };

// One STAGE = one round of up to SF_STAGE_TICKS ticks of the block's group of envs. What it needs is split by writer:
//  * SfStagePrep: the records, the round's stroke list and control values, written by the stepping warp before the stage
//    is handed to the drawing warps and only read after that. A ring of SF_PREP_SLOTS: stage s is prepared in slot
//    s % SF_PREP_SLOTS, so warp 0 can be up to SF_PREP_SLOTS - 1 stages ahead of the stage being drawn.
//  * SfStagePool: what the drawing warps write while they draw a stage (regions, coverage cells, explosion build
//    scratch, work counters). One copy: stages are drawn one after the other.
#ifndef SF_PREP_SLOTS
#define SF_PREP_SLOTS 3   // 2: warp 0 prepares stage s + 1 while stage s is drawn; 3: up to s + 2
#endif
static_assert(SF_PREP_SLOTS >= 2 && SF_PREP_SLOTS <= 6, "named barriers 3 .. 3 + 2 * SF_PREP_SLOTS - 1 must exist (16 per block)");
// Ring of the block's next group ids (rollout kernel), indexed by the block's group count. Warp 0 writes the entry of
// group j when it starts preparing j; the drawing warps read the entry of group g after their last stage of g. Warp 0 can
// only have passed the wait for stage s - 1 - SF_PREP_SLOTS when it starts group j at stage s, so the readers of the groups
// from j - 1 - SF_PREP_SLOTS on may still be pending: the ring needs more than SF_PREP_SLOTS + 1 entries.
#define SF_NEXT_GROUPS 8
static_assert(SF_PREP_SLOTS + 2 <= SF_NEXT_GROUPS, "next-group ring too small for the lead of the stepping warp");
struct __align__(16) SfStagePrep {
  SfEnvRec env[SF_STAGE_SLOTS];
  SfStrokeRec stroke[SF_ROUND_STROKES];
  int r0, r1, nstrokes, build_env;   // the current round: env slots [r0, r1), strokes in the list, the env slot whose explosion is built (-1)
  int netask, chunk, more, nticks;   // env tasks of the round; strokes per batch of phase B1; env slots of the stage are left for
                                     // another round; ticks the stage covers (1 .. SF_STAGE_TICKS)
  int build_env2, padp[3];
  unsigned short etask[SF_STAGE_SLOTS * 5];  // env slot | kind<<6: kind 0..3 = quarter of a dead ship's explosion box, 4 = score strip
};
struct __align__(16) SfStagePool {
  int4 region[SF_POOL_REGIONS];      // {x0, y0, w | h<<16, first cell | tag<<15 | colour<<16}
  short stroke_region[SF_ROUND_STROKES];  // region of stroke k of the round's list, -1: none
  int next_task, next_patch, nregions, cells_used;  // phase C work queue; base patches handed out; regions / cells opened
  int base_ready, padq[3];                          // the round's bulk copies have landed (set by the warp that issued them)
  unsigned short exp_item0[SF_EXP_QUADS];   // build: copies of the y phase's per-quad table entries (SfExpPhase) for the sprite pass
  short exp_qxmin[SF_EXP_QUADS];
  signed char exp_row0[SF_EXP_QUADS];
  unsigned short exp_len[SF_EXPT_ITEMS][SF_EXPT_NC];  // build: summed span lengths of the (quad, pixel row) items of the explosion, per cell
  alignas(16) unsigned arc_mask[SF_EXP_W * SF_EXP_W][4];  // build: per pixel of the explosion box, the quads that cover it (zero between builds)
  alignas(16) unsigned short cells[SF_POOL_CELLS];  // coverage of every region of the round, zero between rounds
};

// The scalar state of the block's group between the ticks of one launch (rollout kernel, warp 0 only): loaded from the SoA
// arrays at the group's first tick, written back at its last one. In between the stepping warp exchanges 112 bytes per env
// with shared memory instead of issuing 7 global loads and 7 global stores per tick into the memory pipeline that the 23
// drawing warps keep full (measured: 4.1 k + 7.0 k of its 27 k cycles per tick went there).
struct __align__(16) SfStepSmem {
  double2 pos[SF_GROUP_ENVS], vel[SF_GROUP_ENVS];
  int4 q0[SF_GROUP_ENVS], q1[SF_GROUP_ENVS], q2[SF_GROUP_ENVS], q3[SF_GROUP_ENVS], st3[SF_GROUP_ENVS];
  unsigned d0[SF_GROUP_ENVS], d1[SF_GROUP_ENVS], d2[SF_GROUP_ENVS];  // pending Stats increments (8-bit fields, flushed every 8 ticks)
};

// per-block shared memory: copies of the static tables that every window touches, and the teams
struct __align__(16) SfBlockSmem {
  int4 xtap[84];   // INTER_AREA taps {si | cnt<<8, a0, a1, a2} (float bits) for the 84 output columns / rows
  int4 ytap[84];
  alignas(16) unsigned char bg_obs[84 * 84];                 // default observation: source of the bulk chunk stores
  alignas(16) unsigned char bg_nat[SF_NAT_H * SF_NAT_STRIDE];  // hexagons on black, native
  unsigned char col_out0[SF_NAT_W + 2], col_out1[SF_NAT_W + 2], row_out0[SF_NAT_H], row_out1[SF_NAT_H];  // native -> output footprint
  unsigned char fort_rect[SF_FORT_STATES][4];
  unsigned short fort_list_xy[36][SF_FORT_LIST_SMEM];  // lit pixels of the fortress sprites (native x | y<<8) ...
  unsigned char fort_list_a[36][SF_FORT_LIST_SMEM];    // ... and their coverage; 0 pads the tail (a blend with alpha 0 changes nothing)
  unsigned char fort_list_n[36];
  unsigned char fort_sparse[SF_FORT_STATES][16];  // first 16 chunks a fortress state changes (255: none); a live fortress changes <= 14
  alignas(16) unsigned magic[SF_MAGIC_N];      // scan converter reciprocals
  alignas(16) SfHot hot;                       // cos / sin of integer degrees (host libm), hexagons, atan2 octants: read by the step too
  double wf_line[3][4][4];                     // wireframe models
  int wf_nlines[4];
  unsigned colour_white, padc[3];
  unsigned char exp_colour[SF_EXP_STROKES + 3];
  alignas(16) unsigned long long init_mbar, pad_mbar;  // the bulk copy of the static part above signals this mbarrier
  int next_group[SF_NEXT_GROUPS];  // rollout kernel: the block's next groups (written by warp 0 ahead of the drawing warps)
  SfStepSmem step;             // rollout kernel: the group's scalar state between ticks
  SfStagePrep prep[SF_PREP_SLOTS];
  SfStagePool pool;
};

// Everything above `init_mbar` is static (a function of the tables only). sf_pack_static_kernel builds it once per
// handle with sf_block_smem_fill and leaves an image in global memory (SfDev::static_image); every rendering block then
// fetches the image with ONE bulk copy (cp.async.bulk global -> shared, completion on an mbarrier) instead of ~25 strided
// loads per thread, while its threads zero the pools (tables ready 1.3 us after block start instead of 5.5 us).
#define SF_STATIC_BYTES ((offsetof(SfBlockSmem, init_mbar) + 15) & ~(size_t)15)

// all kernels that render use the same dynamic shared array: one SfBlockSmem, then one SfWarpSmem per warp.
// Helpers that are kept out of line re-derive their slots from it, so the compiler still knows the address space.
extern __shared__ __align__(16) unsigned char sf_smem_raw[];
__device__ __forceinline__ SfBlockSmem& sf_block_smem() { return *reinterpret_cast<SfBlockSmem*>(sf_smem_raw); }
__device__ __forceinline__ SfStagePrep& sf_prep(int sg) { return sf_block_smem().prep[sg]; }  // sg: the ring slot of the stage being drawn, handed down in a register
__device__ __forceinline__ SfStagePool& sf_pool() { return sf_block_smem().pool; }
// Hand-over of ring slot i between the two roles: two named hardware barriers of 768 threads each, full[i] = 3 + i and
// empty[i] = 3 + SF_PREP_SLOTS + i (bar 0: __syncthreads, bar 2: the drawing warps).
//  * full[i]: warp 0 ARRIVES when it has written the stage into slot i; the 23 drawing warps SYNC on it before they read it.
//  * empty[i]: the drawing warps ARRIVE when they have drawn the stage in slot i; warp 0 SYNCS on it before it rewrites it.
// Memory ordering (PTX memory model, CTA scope): bar.arrive is a release of everything the arriving thread wrote or read
// before it, and bar.sync is an acquire of what the threads that arrived at the same barrier instance released. So the
// records warp 0 wrote are visible to every drawing warp that returns from full[i], and every read of the slot by a
// drawing warp is done before warp 0 returns from empty[i] and overwrites it. Nobody polls: a warp that waits sleeps in
// the barrier. A barrier instance is reused only after it completed: warp 0 arrives at full[i] again (stage s + N) only
// after its sync on empty[i], which needs the drawing warps' arrival after stage s, which followed their sync on full[i]
// for stage s; the same chain orders two uses of empty[i]. Since the drawing warps draw the stages in order and all of
// them sync on full[i], that barrier also separates the pool use of one stage from the next (see sf_drawer_ticks).
__device__ __forceinline__ void sf_stage_full_arrive(int sg) {  // warp 0
  asm volatile("bar.arrive %0, %1;" :: "r"(3 + sg), "r"(32 * SF_RENDER_WARPS) : "memory");
}
__device__ __forceinline__ void sf_stage_full_wait(int sg) {  // drawing warps
  SF_BT_BEGIN();
  asm volatile("bar.sync %0, %1;" :: "r"(3 + sg), "r"(32 * SF_RENDER_WARPS) : "memory");
  SF_BT(0);
}
__device__ __forceinline__ void sf_stage_empty_arrive(int sg) {  // drawing warps
  asm volatile("bar.arrive %0, %1;" :: "r"(3 + SF_PREP_SLOTS + sg), "r"(32 * SF_RENDER_WARPS) : "memory");
}
__device__ __forceinline__ void sf_stage_empty_wait(int sg) {  // warp 0
  SF_BT_BEGIN();
  asm volatile("bar.sync %0, %1;" :: "r"(3 + SF_PREP_SLOTS + sg), "r"(32 * SF_RENDER_WARPS) : "memory");
  SF_BT(2);
}
__device__ __forceinline__ void sf_render_sync() {  // the warps that draw: all but warp 0, which steps (named barrier 2)
  SF_BT_BEGIN();
  asm volatile("bar.sync 2, %0;" :: "r"(32 * (SF_RENDER_WARPS - 1)) : "memory");
  SF_BT(1);
}
__device__ __forceinline__ SfWarpSmem& sf_warp_smem(int warp) { return reinterpret_cast<SfWarpSmem*>(sf_smem_raw + sizeof(SfBlockSmem))[warp]; }
__device__ __forceinline__ SfWarpSmem& sf_my_smem() { return sf_warp_smem(threadIdx.x >> 5); }
#define SF_RENDER_SMEM_BYTES(warps) (sizeof(SfBlockSmem) + sizeof(SfWarpSmem) * (warps))

__device__ __forceinline__ int sf_warp_min(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int sf_warp_max(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int sf_div_small(int a, int b, float inv_b) {  // a / b for 0 <= a < 2^20, exact
  return __float2int_rz(((float)a + 0.5f) * inv_b);
}
__device__ __forceinline__ int sf_div15(int d) { return (d * 2185) >> 15; }  // exact for 0 <= d < 4694

// The static part of SfBlockSmem from the tables (every thread of the block; no barrier inside).
__device__ __forceinline__ void sf_block_smem_fill(const SfTables* T) {
  SfBlockSmem& B = sf_block_smem();
  for (int k = threadIdx.x; k < 168; k += blockDim.x) {
    const SfTap t = k < 84 ? T->xtap[k] : T->ytap[k - 84];
    int4 v = make_int4(t.si | (t.cnt << 8), __float_as_int(t.a[0]), __float_as_int(t.a[1]), __float_as_int(t.a[2]));
    if (k < 84) B.xtap[k] = v; else B.ytap[k - 84] = v;
  }
  for (int k = threadIdx.x; k < 84 * 84 / 16; k += blockDim.x) reinterpret_cast<int4*>(B.bg_obs)[k] = __ldg(reinterpret_cast<const int4*>(T->bg_obs) + k);
  for (int k = threadIdx.x; k < SF_NAT_H * SF_NAT_STRIDE / 16; k += blockDim.x) reinterpret_cast<int4*>(B.bg_nat)[k] = __ldg(reinterpret_cast<const int4*>(T->bg_nat) + k);
  for (int k = threadIdx.x; k < SF_NAT_W + 2; k += blockDim.x) { B.col_out0[k] = k < SF_NAT_W ? (unsigned char)T->col_out0[k] : 0; B.col_out1[k] = k < SF_NAT_W ? (unsigned char)T->col_out1[k] : 0; }
  for (int k = threadIdx.x; k < SF_NAT_H; k += blockDim.x) { B.row_out0[k] = (unsigned char)T->row_out0[k]; B.row_out1[k] = (unsigned char)T->row_out1[k]; }
  for (int k = threadIdx.x; k < SF_FORT_STATES * 4; k += blockDim.x) B.fort_rect[k >> 2][k & 3] = T->fort_rect[k >> 2][k & 3];
  for (int k = threadIdx.x; k < 36 * SF_FORT_LIST_SMEM; k += blockDim.x) {
    const int st = k / SF_FORT_LIST_SMEM, i = k - st * SF_FORT_LIST_SMEM;
    B.fort_list_xy[st][i] = T->fort_list_xy[st][i]; B.fort_list_a[st][i] = i < T->fort_list_n[st] ? T->fort_list_a[st][i] : 0;
  }
  if (threadIdx.x < 36) B.fort_list_n[threadIdx.x] = (unsigned char)min(T->fort_list_n[threadIdx.x], 255);
  for (int k = threadIdx.x; k < SF_FORT_STATES * 16; k += blockDim.x) B.fort_sparse[k >> 4][k & 15] = T->fort_sparse[k >> 4][k & 15];
  for (int k = threadIdx.x; k < SF_MAGIC_N; k += blockDim.x) B.magic[k] = T->magic[k];
  for (int k = threadIdx.x; k < (int)(sizeof(SfHot) / 16); k += blockDim.x) reinterpret_cast<int4*>(&B.hot)[k] = __ldg(reinterpret_cast<const int4*>(&T->hot) + k);
  for (int k = threadIdx.x; k < 48; k += blockDim.x) (&B.wf_line[0][0][0])[k] = (&T->wf_line[0][0][0])[k];
  if (threadIdx.x < 4) B.wf_nlines[threadIdx.x] = threadIdx.x < 3 ? T->wf_nlines[threadIdx.x] : 0;
  if (threadIdx.x < 4) (&B.colour_white)[threadIdx.x] = threadIdx.x == 0 ? T->colour_white : 0u;
  for (int k = threadIdx.x; k < SF_EXP_STROKES + 3; k += blockDim.x) B.exp_colour[k] = k < SF_EXP_STROKES ? T->exp_colour[k] : 0;
}

// once per block at kernel start (every thread of the block calls it, before any early exit): the static part arrives
// as one bulk copy of the handle's image while the threads zero the pools
// (Tried and dropped: letting warp 0 step the first tick while the other warps load the tables — its first step ran
// slower next to the loads and the extra live state cost the drawing code registers: -3 % overall.)
__device__ __forceinline__ void sf_block_smem_init(const unsigned char* image) {
  SfBlockSmem& B = sf_block_smem();
  SF_TL_START();
  const unsigned bar = (unsigned)__cvta_generic_to_shared(&B.init_mbar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"((unsigned)SF_STATIC_BYTES) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"((unsigned)__cvta_generic_to_shared(&B)), "l"(image), "r"((unsigned)SF_STATIC_BYTES), "r"(bar) : "memory");
  }
  for (int k = threadIdx.x; k < SF_POOL_CELLS / 2; k += blockDim.x) reinterpret_cast<unsigned*>(B.pool.cells)[k] = 0u;
  for (int k = threadIdx.x; k < SF_EXP_W * SF_EXP_W * 4; k += blockDim.x) (&B.pool.arc_mask[0][0])[k] = 0u;
  if (threadIdx.x == 32) { B.pool.next_task = 0; B.pool.next_patch = 0; B.pool.nregions = 0; B.pool.cells_used = 0; B.pool.base_ready = 0; }
  // no env in the ring yet (sf_publish_recs compares a new record with the ones of the rounds before it)
  for (int k = threadIdx.x; k < SF_PREP_SLOTS * SF_STAGE_SLOTS; k += blockDim.x) B.prep[k / SF_STAGE_SLOTS].env[k % SF_STAGE_SLOTS].env = -1;
  // the bulk-copy engine (async proxy) reads bg_obs: make generic-proxy writes visible to it
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();   // (also: the mbarrier is initialised before anybody polls it)
  unsigned ok;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(bar) : "memory");
  } while (!ok);
  SF_TL(2);
}
// once per warp at kernel start
__device__ __forceinline__ void sf_warp_smem_init(SfWarpSmem& W, int lane) {
  if (lane == 0) W.ngroups = 0;
  __syncwarp();
}

// body(c, r) for every 0 <= c < w, 0 <= r < h (w <= 32): narrow rectangles put several rows on one pass
template <class F>
__device__ __forceinline__ void sf_for_rect(int lane, int w, int h, F body) {
  const int s = w <= 8 ? 3 : (w <= 16 ? 4 : 5);
  const int c = lane & ((1 << s) - 1), rstep = 32 >> s;
  if (c < w)
    for (int r = lane >> s; r < h; r += rstep) body(c, r);
}

// the same, as load / store pairs with up to four loads in flight: store(c, r, load(c, r))
template <class L, class S>
__device__ __forceinline__ void sf_for_rect4(int lane, int w, int h, L load, S store) {
  const int s = w <= 8 ? 3 : (w <= 16 ? 4 : 5);
  const int c = lane & ((1 << s) - 1), rstep = 32 >> s;
  if (c < w)
    for (int r = lane >> s; r < h; r += 4 * rstep) {
      const int r1 = r + rstep, r2 = r + 2 * rstep, r3 = r + 3 * rstep;
      auto v0 = load(c, r);
      auto v1 = load(c, r1 < h ? r1 : r), v2 = load(c, r2 < h ? r2 : r), v3 = load(c, r3 < h ? r3 : r);
      store(c, r, v0);
      if (r1 < h) store(c, r1, v1);
      if (r2 < h) store(c, r2, v2);
      if (r3 < h) store(c, r3, v3);
    }
}

// ---- edge records --------------------------------------------------------------------------------------
// An edge from (xa, ga) to (xb, gb), ga < gb grid rows, crosses sub-row s at x(s) = xa + floor((s - ga) * dx / dy).
// The record is referenced to the end where the product is non-negative: dx >= 0: x0 = xa, yref = ga; dx < 0:
// x0 = xb, yref = gb (floor((s-ga)*dx/dy) == dx + floor((gb-s)*|dx|/dy)). Then n = (s - yref) * dx >= 0 always and
// x(s) = x0 + floor(n / dy) = x0 + umulhi(n, M) with the magic reciprocal M = floor((2^32-1)/dy) + 1 (exact while
// n * dy < 2^32: always true for the strokes drawn here, at most ~30 px tall and ~10 px wide).
__device__ __forceinline__ int4 sf_make_edge(const SfTables* T, int xa, int ga, int xb, int gb) {  // ga < gb
  const int dy = gb - ga, dx = xb - xa;
  const unsigned M = sf_block_smem().magic[min(dy, SF_MAGIC_N - 1)];  // device strokes are far shorter than 512 sub-rows (34 px)
  const int a = ga + SF_YBIAS, b = gb + SF_YBIAS;
  if (dy == 1) return make_int4(xa, a | (b << 16), 0, 0);  // one sample, at the top row: x = xa (2^32/1 has no 32-bit magic)
  return dx >= 0 ? make_int4(xa, a | (b << 16), dx, (int)M) : make_int4(xb, b | (a << 16), dx, (int)M);
}
__device__ __forceinline__ int sf_edge_x(int4 E, int sb) {  // sb = s + bias inside the edge's rows
  return E.x + (int)__umulhi((unsigned)((sb - (E.y & 0xFFFF)) * E.z), (unsigned)E.w);
}

// what the lane that built a quad knows about it
struct SfQuadGeom {
  int ymin_g, ymax_g, xmin, xmax;  // bounding box (grid rows / 24.8 x); ymin_g >= ymax_g: covers no sample
  int split;                       // first (biased) sub-row of the second down edge | second up edge << 16
  int flags;                       // SF_QF_IRREGULAR
};

// Build the 4 edge records of convex quad q (cyclic corners, consistent orientation) into slot `qi`.
// Edges whose grid rows increase along the traversal lie on one side, the others on the opposite side; a stroked
// segment is a parallelogram, so each side has at most two non-degenerate edges. Trapezoids (explosion arcs that
// straddle 0/180 degrees) can have three on one side: those keep all edges and the span tests every one.
__device__ __noinline__ void sf_store_quad_edges(const SfTables* T, int qi, int x0, int y0, int x1, int y1, int x2, int y2, int x3, int y3,
                                                  SfQuadGeom& G) {
  SfWarpSmem& W = sf_my_smem();
  const int g0 = sf_grid_y(y0), g1 = sf_grid_y(y1), g2 = sf_grid_y(y2), g3 = sf_grid_y(y3);
  const int4 none = make_int4(0, 0, 0, 0);  // yref == yother: never live
  int4 E0 = none, E1 = none, E2 = none, E3 = none;
  int d0 = 0, d1 = 0, d2 = 0, d3 = 0;  // +1: rows increase along the traversal, -1: decrease, 0: degenerate
  if (g0 < g1) { E0 = sf_make_edge(T, x0, g0, x1, g1); d0 = 1; } else if (g0 > g1) { E0 = sf_make_edge(T, x1, g1, x0, g0); d0 = -1; }
  if (g1 < g2) { E1 = sf_make_edge(T, x1, g1, x2, g2); d1 = 1; } else if (g1 > g2) { E1 = sf_make_edge(T, x2, g2, x1, g1); d1 = -1; }
  if (g2 < g3) { E2 = sf_make_edge(T, x2, g2, x3, g3); d2 = 1; } else if (g2 > g3) { E2 = sf_make_edge(T, x3, g3, x2, g2); d2 = -1; }
  if (g3 < g0) { E3 = sf_make_edge(T, x3, g3, x0, g0); d3 = 1; } else if (g3 > g0) { E3 = sf_make_edge(T, x0, g0, x3, g3); d3 = -1; }
  const int nd = (d0 > 0) + (d1 > 0) + (d2 > 0) + (d3 > 0), nu = (d0 < 0) + (d1 < 0) + (d2 < 0) + (d3 < 0);
  const int gmin = min(min(g0, g1), min(g2, g3)), gmax = max(max(g0, g1), max(g2, g3));
  G.flags = 0; G.split = 0;
  if (nd == 0 || nu == 0) { G.ymin_g = 1 << 30; G.ymax_g = -(1 << 30); G.xmin = 1 << 30; G.xmax = -(1 << 30); return; }
  if (nd > 2 || nu > 2) {
    W.edge[qi * 4 + 0] = E0; W.edge[qi * 4 + 1] = E1; W.edge[qi * 4 + 2] = E2; W.edge[qi * 4 + 3] = E3;
    G.flags = SF_QF_IRREGULAR;
  } else {
    // first / second edge of each direction in cyclic order, with the (biased) top row of each
    auto top = [](int4 E) { return min(E.y & 0xFFFF, (int)((unsigned)E.y >> 16)); };
    int4 dnA = d0 > 0 ? E0 : d1 > 0 ? E1 : d2 > 0 ? E2 : E3;
    int4 dnB = d3 > 0 ? E3 : d2 > 0 ? E2 : d1 > 0 ? E1 : E0;
    int4 upA = d0 < 0 ? E0 : d1 < 0 ? E1 : d2 < 0 ? E2 : E3;
    int4 upB = d3 < 0 ? E3 : d2 < 0 ? E2 : d1 < 0 ? E1 : E0;
    // order each side top to bottom; a side with one edge has A == B (the split test selects B, same edge)
    if (top(dnB) < top(dnA)) { int4 t = dnA; dnA = dnB; dnB = t; }
    if (top(upB) < top(upA)) { int4 t = upA; upA = upB; upB = t; }
    W.edge[qi * 4 + 0] = dnA; W.edge[qi * 4 + 1] = dnB; W.edge[qi * 4 + 2] = upA; W.edge[qi * 4 + 3] = upB;
    G.split = top(dnB) | (top(upB) << 16);
  }
  G.ymin_g = gmin; G.ymax_g = gmax;
  G.xmin = min(min(x0, x1), min(x2, x3)); G.xmax = max(max(x0, x1), max(x2, x3));
}

// ---- batch machinery ---------------------------------------------------------------------------------------
// The block owns the region list and the coverage cells of a round; a warp owns the edge / quad / stroke records
// of the batch it is scan-converting.

// floor division of a grid row by 15
__device__ __forceinline__ int sf_row_of(int g) { return (g >= 0) ? g / SF_GRID_Y : -((-g + SF_GRID_Y - 1) / SF_GRID_Y); }

// Append one region per participating lane (`want`) to the block's list, in lane order: region ids and coverage
// cells come from the block-wide pools (one atomic per batch each). Returns the lane's region id, or -1 when the
// stroke is off the surface (or a pool is full: cannot happen, the round scan admits envs by worst-case need).
__device__ __forceinline__ int sf_open_regions(int lane, bool want, int ymin_g, int ymax_g, int xmin, int xmax, unsigned colour, int tag) {
  SfStagePool& Tm = sf_pool();
  int cx0 = 0, py0 = 0, w = 0, h = 0;
  bool ok = want && ymin_g < ymax_g;
  if (ok) {
    py0 = max(sf_row_of(ymin_g), 0); int py1 = min(sf_row_of(ymax_g - 1), SF_NAT_H - 1);
    cx0 = max(xmin >> 8, 0); int cx1 = min((xmax - 1) >> 8, SF_NAT_W - 1);
    ok = py0 <= py1 && cx0 <= cx1;
    w = cx1 - cx0 + 1; h = py1 - py0 + 1;
    if (w > 255 || h > 255) ok = false;
  }
  const int cells = ok ? w * h : 0;
  int incl = cells;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  const unsigned okmask = __ballot_sync(0xffffffffu, ok);
  int base_c = 0, base_r = 0;
  if (lane == 31) { base_c = atomicAdd(&Tm.cells_used, incl); base_r = atomicAdd(&Tm.nregions, __popc(okmask)); }
  base_c = __shfl_sync(0xffffffffu, base_c, 31); base_r = __shfl_sync(0xffffffffu, base_r, 31);
  const int rid = base_r + __popc(okmask & ((1u << lane) - 1u));
  if (ok && (base_c + incl > SF_POOL_CELLS || rid >= SF_POOL_REGIONS)) ok = false;
  if (!ok) return -1;
  Tm.region[rid] = make_int4(cx0, py0, w | (h << 16), (base_c + incl - cells) | (tag << 15) | ((int)colour << 16));
  return rid;
}

// Publish the batch for the scan converter. Every lane that built a quad (`has`) stores its live sub-rows clipped to
// the region of its stroke; the first lane of every stroke slot (`head`: nq consecutive lanes starting here hold the
// quads of the stroke, [s0, s1) = union of their live sub-rows) stores the stroke record and appends the stroke's
// work groups of 8 consecutive sub-rows. rid = the stroke's region (-1: none).
__device__ __forceinline__ void sf_publish_quads(SfWarpSmem& W, int lane, const SfQuadGeom& G, bool has, int rid, bool head, int slot, int nq, int ymin_g, int ymax_g) {
  const SfStagePool& Tm = sf_pool();
  int len = 0;
  int4 R = make_int4(0, 0, 0, 0);
  if (rid >= 0) R = Tm.region[rid];
  const int w = R.z & 0xFFFF, h = (R.z >> 16) & 0xFFFF;
  const int top = R.y * SF_GRID_Y + SF_YBIAS;
  if (has && rid >= 0) {
    const int g0 = max(G.ymin_g + SF_YBIAS, top), g1 = min(G.ymax_g + SF_YBIAS, top + h * SF_GRID_Y);
    W.qinfo[lane] = make_int4(g0 | (max(g1, g0) << 16), G.split, G.flags, 0);
  } else W.qinfo[lane] = make_int4(0, 0, 0, 0);  // g0 == g1: never live
  if (head && rid >= 0) {
    const int s0 = max(ymin_g + SF_YBIAS, top), s1 = min(ymax_g + SF_YBIAS, top + h * SF_GRID_Y);
    len = max(s1 - s0, 0);
    W.srec[slot] = make_int4(R.x | (w << 8) | (nq << 16) | (lane << 24), top, R.w & 0x7FFF, s0 | (max(s1, s0) << 16));
  }
  // work groups of 8 consecutive sub-rows
  const int n8 = (len + 7) >> 3;
  int gs = n8;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, gs, o); if (lane >= o) gs += t; }
  const int total = __shfl_sync(0xffffffffu, gs, 31);
  gs -= n8;
  for (int k = 0; k < n8; k++)
    if (gs + k < SF_MAX_GROUPS) W.glist[gs + k] = (unsigned short)(slot | (k << 5));
  if (lane == 0) W.ngroups = min(total, SF_MAX_GROUPS);
  __syncwarp();
}

// Span of quad q (a stroked segment: a parallelogram, opposite edges run in opposite directions, so each side has at
// most two edges) on sub-row sb, clipped to [xlo, xhi) and made relative to xlo, packed lo<<16 | hi; SF_SPAN_NONE when
// the quad has no sample there. Branch free: the loads of all quads of a stroke can be in flight together. A quad
// slot without a quad has g0 == g1 (never live); whatever its edge records hold is evaluated and discarded.
__device__ __forceinline__ unsigned sf_quad_span_regular(const SfWarpSmem& W, int q, int sb, int xlo, int xhi) {
  const int4 Q = W.qinfo[q];
  const int4 Ed = W.edge[q * 4 + (sb >= (Q.y & 0xFFFF) ? 1 : 0)];
  const int4 Eu = W.edge[q * 4 + 2 + (sb >= (int)((unsigned)Q.y >> 16) ? 1 : 0)];
  const int xd = sf_edge_x(Ed, sb), xu = sf_edge_x(Eu, sb);
  const int lo = max(min(xd, xu), xlo) - xlo, hi = min(max(xd, xu), xhi) - xlo;
  const bool live = sb >= (Q.x & 0xFFFF) && sb < (int)((unsigned)Q.x >> 16) && lo < hi;
  return live ? (((unsigned)lo << 16) | (unsigned)hi) : SF_SPAN_NONE;
}

// Scan-convert the batch: one lane per (stroke, sub-row). The lane computes the exact span of every quad of the
// stroke that is live on its sub-row (integer edge stepping), sorts the <= 4 spans and adds each one minus the
// union of its predecessors to the coverage cells of the stroke's region (non-zero winding of equally oriented
// convex quads == union). 8 lanes share a work group of 8 consecutive sub-rows of one stroke.
__device__ __forceinline__ void sf_emit_span_pred(unsigned* acc32, int cell0, int a, int b) {
  // straight-line version of sf_emit_span: the two partial cells are predicated, only the run of full cells in
  // between (near-horizontal spans) loops
  const bool any = a < b;
  const int c1 = a >> 8, c2 = (b - 1) >> 8;
  const int ci = cell0 + c1, cj = cell0 + c2;
  const unsigned len1 = (unsigned)(min(b, (c1 + 1) << 8) - a), len2 = (unsigned)(b - (c2 << 8));
  if (any) atomicAdd(&acc32[ci >> 1], len1 << ((ci & 1) << 4));
  if (any && c2 > c1) atomicAdd(&acc32[cj >> 1], len2 << ((cj & 1) << 4));
  if (any && c2 > c1 + 1)
    for (int c = c1 + 1; c < c2; c++) { const int cm = cell0 + c; atomicAdd(&acc32[cm >> 1], 256u << ((cm & 1) << 4)); }
}

// One pass (4 work groups = 32 (stroke, sub-row) items) of the batch that warp `owner` published, starting at its
// work group g0. Any warp of the block can run any pass: the records are read-only after the block barrier that
// follows the geometry, and the cells are updated with atomics.
__device__ __noinline__ void sf_accumulate_pass(int owner, int g0) {
  const SfWarpSmem& W = sf_warp_smem(owner);
  const int lane = threadIdx.x & 31;
  const int ngroups = W.ngroups;
  unsigned* acc32 = reinterpret_cast<unsigned*>(sf_pool().cells);
  const int gi = min(g0 + (lane >> 3), ngroups - 1);
  const int ent = W.glist[gi];
  const int4 S = W.srec[ent & 31];
  const int sb = (S.w & 0xFFFF) + ((ent >> 5) << 3) + (lane & 7);
  const bool valid = g0 + (lane >> 3) < ngroups && sb < (int)((unsigned)S.w >> 16);
  const int q0 = (int)((unsigned)S.x >> 24);
  const int w = (S.x >> 8) & 255;
  const int xlo = (S.x & 255) << 8, xhi = xlo + (w << 8);
  const int cell0 = S.z + sf_div15(max(sb - S.y, 0)) * w;
  // wireframes: 3 or 4 stroked segments (a slot without a quad is never live); all loads in flight together
  unsigned k0 = sf_quad_span_regular(W, q0, sb, xlo, xhi);
  unsigned k1 = sf_quad_span_regular(W, q0 + 1, sb, xlo, xhi);
  unsigned k2 = sf_quad_span_regular(W, q0 + 2, sb, xlo, xhi);
  unsigned k3 = SF_SPAN_NONE;
  if (__any_sync(0xffffffffu, ((S.x >> 16) & 255) > 3)) k3 = sf_quad_span_regular(W, q0 + 3, sb, xlo, xhi);  // only shells have a 4th segment
  if (!valid) { k0 = SF_SPAN_NONE; k1 = SF_SPAN_NONE; k2 = SF_SPAN_NONE; k3 = SF_SPAN_NONE; }
  // sort by start (none == 0xFFFFFFFF sinks to the end)
  unsigned t0 = min(k0, k1), t1 = max(k0, k1), t2 = min(k2, k3), t3 = max(k2, k3);
  k0 = min(t0, t2); k2 = max(t0, t2);
  k1 = min(t1, t3); k3 = max(t1, t3);
  t0 = min(k1, k2); k2 = max(k1, k2); k1 = t0;
  // each span minus the union of its predecessors; none: a = 0xFFFF > b
  int reach = 0;
  { const int a = (int)(k0 >> 16), b = k0 == SF_SPAN_NONE ? 0 : (int)(k0 & 0xFFFFu); sf_emit_span_pred(acc32, cell0, a, b); reach = b; }
  { const int a = max((int)(k1 >> 16), reach), b = k1 == SF_SPAN_NONE ? 0 : (int)(k1 & 0xFFFFu); sf_emit_span_pred(acc32, cell0, a, b); reach = max(reach, b); }
  { const int a = max((int)(k2 >> 16), reach), b = k2 == SF_SPAN_NONE ? 0 : (int)(k2 & 0xFFFFu); sf_emit_span_pred(acc32, cell0, a, b); reach = max(reach, b); }
  { const int a = max((int)(k3 >> 16), reach), b = k3 == SF_SPAN_NONE ? 0 : (int)(k3 & 0xFFFFu); sf_emit_span_pred(acc32, cell0, a, b); }
}

// ---- windows ---------------------------------------------------------------------------------------------
// win = nx0 | ny0<<8 | pw<<16 | ph<<24 : native rectangle held in W.patch (row stride 32)
#define SF_WIN_X0(win) ((win) & 255)
#define SF_WIN_Y0(win) (((win) >> 8) & 255)
#define SF_WIN_W(win) (((win) >> 16) & 255)
#define SF_WIN_H(win) (((unsigned)(win)) >> 24)

__device__ __forceinline__ void sf_patch_init(SfWarpSmem& W, const SfTables* T, int lane, int win) {
  const int nx0 = SF_WIN_X0(win), ny0 = SF_WIN_Y0(win);
  const unsigned char* bg = sf_block_smem().bg_nat + ny0 * SF_NAT_STRIDE + nx0;
  sf_for_rect(lane, SF_WIN_W(win), SF_WIN_H(win), [&](int c, int r) { W.patch[r * SF_PATCH_STRIDE + c] = bg[r * SF_NAT_STRIDE + c]; });
  __syncwarp();
}

// Blend region `rid` of the round (its coverage cells) into this warp's window (clipped to it).
__device__ __noinline__ void sf_blend_region(int rid, int win) {
  SfWarpSmem& W = sf_my_smem();
  const SfStagePool& O = sf_pool();
  const int lane = threadIdx.x & 31;
  const int4 R = O.region[rid];
  const int w = R.z & 0xFFFF, h = (R.z >> 16) & 0xFFFF;
  const int nx0 = SF_WIN_X0(win), ny0 = SF_WIN_Y0(win);
  const int ix0 = max(R.x, nx0), ix1 = min(R.x + w, nx0 + SF_WIN_W(win));
  const int iy0 = max(R.y, ny0), iy1 = min(R.y + h, ny0 + (int)SF_WIN_H(win));
  if (ix0 >= ix1 || iy0 >= iy1) return;
  const unsigned colour = ((unsigned)R.w >> 16) & 255u;
  const unsigned short* cells = O.cells + (R.w & 0x7FFF) + (iy0 - R.y) * w + (ix0 - R.x);
  unsigned char* p0 = W.patch + (iy0 - ny0) * SF_PATCH_STRIDE + (ix0 - nx0);
  sf_for_rect(lane, ix1 - ix0, iy1 - iy0, [&](int c, int r) {
    unsigned L = cells[r * w + c];
    if (L) {
      unsigned char* px = p0 + r * SF_PATCH_STRIDE + c;
      *px = (unsigned char)sf_blend(*px, colour, sf_len_to_alpha(L));
    }
  });
  __syncwarp();
}

// Composite every layer of env slot `e` that intersects the window, in draw order (draw.cpp:227-269), into W.patch.
// Returns true when no wireframe of the env reaches into the window.
__device__ __noinline__ bool sf_composite(const SfTables* T, unsigned char* expcache, int e, int win, int sg) {
  SfWarpSmem& W = sf_my_smem();
  const SfBlockSmem& B = sf_block_smem();
  const SfEnvRec& rec = sf_prep(sg).env[e];
  const int lane = threadIdx.x & 31;
  const unsigned core = rec.core;
  const int nx0 = SF_WIN_X0(win), ny0 = SF_WIN_Y0(win);
  const int nx1 = nx0 + SF_WIN_W(win), ny1 = ny0 + (int)SF_WIN_H(win);  // exclusive
  sf_patch_init(W, T, lane, win);
  // regions of this env (one per visible stroke, in draw order) that reach into the window
  int sr = -1, tag = SF_TAG_PROJECTILE;
  bool hit = false;
  if (lane < rec.ns) {
    sr = sf_pool().stroke_region[rec.s0 + lane];
    if (sr >= 0) {
      const int4 R = sf_pool().region[sr];
      hit = R.x < nx1 && R.x + (R.z & 0xFFFF) > nx0 && R.y < ny1 && R.y + ((R.z >> 16) & 0xFFFF) > ny0;
      tag = (R.w >> 15) & 1;
    }
  }
  unsigned rmask = __ballot_sync(0xffffffffu, hit);
  const bool no_wireframe = rmask == 0u;
  const bool first_is_ship = __shfl_sync(0xffffffffu, tag, 0) == SF_TAG_SHIP;
  // ---- ship wireframe | ship explosion (draw.cpp:233-237) ----
  if (core & SF_CORE_SHIP_ALIVE) {
    if ((rmask & 1u) && first_is_ship) { const int s0r = __shfl_sync(0xffffffffu, sr, 0); sf_blend_region(s0r, win); rmask &= ~1u; }
  } else {
    const int ebox = rec.ebox;
    const int bx0 = (ebox & 255) - 64, by0 = ((ebox >> 8) & 255) - 64;
    const int ix0 = max(max(bx0, 0), nx0), ix1 = min(min(bx0 + SF_EXP_W, SF_NAT_W), nx1);
    const int iy0 = max(max(by0, 0), ny0), iy1 = min(min(by0 + SF_EXP_W, SF_NAT_H), ny1);
    if (ix0 < ix1 && iy0 < iy1) {
      {
        // cached sprite: whole 28-byte rows as 32-bit words, all loads in flight before the first use
        const unsigned* src32 = reinterpret_cast<const unsigned*>(expcache + (iy0 - by0) * SF_EXP_W);
        const int nw = (SF_EXP_W / 4) * (iy1 - iy0);
        unsigned v[7];
#pragma unroll
        for (int u = 0; u < 7; u++) v[u] = lane + 32 * u < nw ? __ldcg(&src32[lane + 32 * u]) : 0u;
#pragma unroll
        for (int u = 0; u < 7; u++) {
          const int k = lane + 32 * u;
          if (k < nw) {
            const int row = (k * 9363) >> 16, x4 = bx0 + (k - row * (SF_EXP_W / 4)) * 4;  // k / 7, exact for k < 196
            unsigned char* dst = W.patch + (iy0 + row - ny0) * SF_PATCH_STRIDE - nx0;
#pragma unroll
            for (int b = 0; b < 4; b++)
              if (x4 + b >= ix0 && x4 + b < ix1) dst[x4 + b] = (unsigned char)(v[u] >> (8 * b));
          }
        }
      }
      __syncwarp();
    }
  }
  // ---- fortress wireframe | fortress explosion (draw.cpp:238-242) ----
  {
    const int fst = (core & SF_CORE_FORT_ALIVE) ? (int)((core >> SF_CORE_FANG_SHIFT) & 63u) : 36;
    const unsigned char* fr = B.fort_rect[fst];
    if ((int)fr[0] < nx1 && (int)fr[2] >= nx0 && (int)fr[1] < ny1 && (int)fr[3] >= ny0) {
      if (fst < 36) {
        const int n = B.fort_list_n[fst];
        const bool in_smem = n <= SF_FORT_LIST_SMEM;  // always, for the sprites of the reference's fortress
#pragma unroll 1
        for (int k = lane; k < n; k += 32) {
          const int xy = in_smem ? B.fort_list_xy[fst][k] : T->fort_list_xy[fst][k];
          const unsigned a = in_smem ? B.fort_list_a[fst][k] : T->fort_list_a[fst][k];
          const int x = xy & 255, y = xy >> 8;
          if (x >= nx0 && x < nx1 && y >= ny0 && y < ny1) {
            unsigned char* px = &W.patch[(y - ny0) * SF_PATCH_STRIDE + (x - nx0)];
            *px = (unsigned char)sf_blend(*px, B.colour_white, a);
          }
        }
      } else {
        const int ix0 = max(SF_FEXP_X0, nx0), ix1 = min(SF_FEXP_X0 + SF_EXP_W, nx1);
        const int iy0 = max(SF_FEXP_Y0, ny0), iy1 = min(SF_FEXP_Y0 + SF_EXP_W, ny1);
        if (ix0 < ix1 && iy0 < iy1) {
          sf_for_rect(lane, ix1 - ix0, iy1 - iy0, [&](int c, int r) {
            const int idx = (iy0 + r - SF_FEXP_Y0) * SF_EXP_W + (ix0 + c - SF_FEXP_X0);
            unsigned a0 = T->fexp_alpha[0][idx];
            if (a0) {
              unsigned char* px = &W.patch[(iy0 + r - ny0) * SF_PATCH_STRIDE + (ix0 + c - nx0)];
              unsigned v = sf_blend(*px, T->fexp_colour[0][idx], a0);
              for (int l = 1; l < T->fexp_layers; l++) {
                unsigned a = T->fexp_alpha[l][idx];
                if (!a) break;
                v = sf_blend(v, T->fexp_colour[l][idx], a);
              }
              *px = (unsigned char)v;
            }
          });
        }
      }
      __syncwarp();
    }
  }
  // ---- missiles, then shells (draw.cpp:243-253): the env's strokes are stored in draw order ----
#pragma unroll 1
  while (rmask) {
    const int q = __ffs(rmask) - 1;
    rmask &= rmask - 1;
    const int sq = __shfl_sync(0xffffffffu, sr, q);
    sf_blend_region(sq, win);
  }
  // ---- score digits (draw.cpp:160-173,267): "%07d" of (int)mPoints ----
  {
    const int ix0 = max(SF_TEXT_X0, nx0), ix1 = min(SF_TEXT_X0 + SF_TEXT_W, nx1);
    const int iy0 = max(SF_TEXT_Y0, ny0), iy1 = min(SF_TEXT_Y0 + SF_TEXT_H, ny1);
    if (ix0 < ix1 && iy0 < iy1) {
      const int pts = min(max(rec.points_i, 0), 9999999);
      sf_for_rect(lane, ix1 - ix0, iy1 - iy0, [&](int c, int r) {
        const int tc = ix0 + c - SF_TEXT_X0, tr = iy0 + r - SF_TEXT_Y0;
        const int slot = T->text_slot[tc];
        if (slot < 7) {
          int div = 1;
          for (int k = slot; k < 6; k++) div *= 10;
          unsigned a = T->text_alpha[(pts / div) % 10][tr * SF_TEXT_W + tc];
          if (a) {
            unsigned char* px = &W.patch[(iy0 + r - ny0) * SF_PATCH_STRIDE + (ix0 + c - nx0)];
            *px = (unsigned char)sf_blend(*px, T->colour_text, a);
          }
        }
      });
      __syncwarp();
    }
  }
  // ---- vulnerability bar (draw.cpp:207-225,268) ----
  {
    const int ix0 = max(SF_BAR_X0, nx0), ix1 = min(SF_BAR_X0 + SF_BAR_W, nx1);
    const int iy0 = max(SF_BAR_Y0, ny0), iy1 = min(SF_BAR_Y0 + SF_BAR_H, ny1);
    if (ix0 < ix1 && iy0 < iy1) {
      const int filled = 4 * min(rec.vuln, 10);  // 20 user units per step = 4 px
      const unsigned fg = rec.kill_bar ? T->colour_bar_kill : T->colour_bar_fg;
      sf_for_rect(lane, ix1 - ix0, iy1 - iy0, [&](int c, int r) {
        const unsigned a = T->bar_alpha[iy0 + r - SF_BAR_Y0];
        unsigned char* px = &W.patch[(iy0 + r - ny0) * SF_PATCH_STRIDE + (ix0 + c - nx0)];
        unsigned v = sf_blend(*px, T->colour_bar_bg, a);
        if (ix0 + c - SF_BAR_X0 < filled) v = sf_blend(v, fg, a);
        *px = (unsigned char)v;
      });
      __syncwarp();
    }
  }
  return no_wireframe;
}

// Resample the window (cv2 INTER_AREA: float accumulation in table order, round-half-even; a missing tap has
// weight +0 and reads a byte of the patch that is never used) and overwrite the output rectangle
// orect = j0 | i0<<8 | ow<<16 | oh<<24.
// `cache` (or NULL): the same pixels also go to the env's resampled explosion box, whose origin is output pixel
// corigin = cj0 | ci0<<8.
__device__ __noinline__ void sf_window_out(int win, int orect, unsigned char* __restrict__ obs84, unsigned char* __restrict__ cache, int corigin) {
  const SfWarpSmem& W = sf_my_smem();
  const SfBlockSmem& B = sf_block_smem();
  const int lane = threadIdx.x & 31;
  const int nx0 = SF_WIN_X0(win), ny0 = SF_WIN_Y0(win);
  const int j0 = orect & 255, i0 = (orect >> 8) & 255;
  sf_for_rect(lane, (orect >> 16) & 255, (int)((unsigned)orect >> 24), [&](int c, int r) {
    const int i = i0 + r, j = j0 + c;
    const int4 tx = B.xtap[j], ty = B.ytap[i];
    const unsigned char* S = &W.patch[((ty.x & 255) - ny0) * SF_PATCH_STRIDE + ((tx.x & 255) - nx0)];
    const float ax0 = __int_as_float(tx.y), ax1 = __int_as_float(tx.z);
    const float b0 = __fadd_rn(__fmul_rn((float)S[0], ax0), __fmul_rn((float)S[1], ax1));
    const float b1 = __fadd_rn(__fmul_rn((float)S[SF_PATCH_STRIDE], ax0), __fmul_rn((float)S[SF_PATCH_STRIDE + 1], ax1));
    const float b2 = __fadd_rn(__fmul_rn((float)S[2 * SF_PATCH_STRIDE], ax0), __fmul_rn((float)S[2 * SF_PATCH_STRIDE + 1], ax1));
    float sum = __fmul_rn(__int_as_float(ty.y), b0);
    sum = __fadd_rn(sum, __fmul_rn(__int_as_float(ty.z), b1));
    sum = __fadd_rn(sum, __fmul_rn(__int_as_float(ty.w), b2));
    const unsigned char v = (unsigned char)__float2int_rn(sum);
    obs84[i * 84 + j] = v;
    if (cache) cache[(i - (corigin >> 8)) * SF_EXPO_STRIDE + (j - (corigin & 255))] = v;
  });
}

// Window of the output rectangle [j0..j1] x [i0..i1] of env slot e: composite its native footprint + resample.
// Returns true when the pixels were also written to `cache` (no wireframe reaches into the window).
__device__ __forceinline__ bool sf_window_orect(const SfTables* T, unsigned char* expcache, int e, int j0, int i0, int j1, int i1, unsigned char* obs84,
                                                unsigned char* cache, int corigin, int sg) {
  const SfBlockSmem& B = sf_block_smem();
  const int tx0 = B.xtap[j0].x, tx1 = B.xtap[j1].x, ty0 = B.ytap[i0].x, ty1 = B.ytap[i1].x;
  const int nx0 = tx0 & 255, nx1 = (tx1 & 255) + (tx1 >> 8) - 1, ny0 = ty0 & 255, ny1 = (ty1 & 255) + (ty1 >> 8) - 1;
  if (nx1 - nx0 + 1 > SF_WIN_MAX_W || ny1 - ny0 + 1 > SF_WIN_MAX_H) __trap();  // no moving box is that large
  const int win = nx0 | (ny0 << 8) | ((nx1 - nx0 + 1) << 16) | ((ny1 - ny0 + 1) << 24);
  const int orect = j0 | (i0 << 8) | ((j1 - j0 + 1) << 16) | ((i1 - i0 + 1) << 24);
  const bool pure = sf_composite(T, expcache, e, win, sg);
  sf_window_out(win, orect, obs84, pure ? cache : nullptr, corigin);
  __syncwarp();
  return pure && cache;
}

// ---- wireframe strokes (R3 drawWireFrame, draw.cpp:82-100) --------------------------------------------------------
// Geometry for up to 8 strokes at once: lane = 4*slot + line. kind: 0 ship, 1 missile, 2 shell, -1 none.
// Every lane passes the description of ITS slot's stroke. Appends one region per visible stroke and publishes the
// quads. Returns the region of the lane's slot (-1 invisible).
__device__ __forceinline__ int sf_wire_geometry(SfWarpSmem& W, int lane, const SfTables* T, int kind, double px, double py, int angle) {
  const int slot = lane >> 2, line = lane & 3;
  SfQuadGeom G;
  G.ymin_g = 1 << 30; G.ymax_g = -(1 << 30); G.xmin = 1 << 30; G.xmax = -(1 << 30); G.split = 0; G.flags = 0;
  bool has = false;
  if (kind >= 0) {
    // quick cull: every model fits in a 37-unit radius (7.4 px) around its origin
    double dxv = SF_DADD(SF_DMUL(px, SF_CTM_SCALE), SF_CTM_X0), dyv = SF_DADD(SF_DMUL(py, SF_CTM_SCALE), SF_CTM_Y0);
    bool visible = !(dxv < -9.0 || dxv > SF_NAT_W + 9.0 || dyv < -9.0 || dyv > SF_NAT_H + 9.0);
    const SfBlockSmem& B = sf_block_smem();
    if (visible && line < B.wf_nlines[kind]) {
      const double2 cs = make_double2(B.hot.cs[angle][0], B.hot.cs[angle][1]);
      SfWireXf m = sf_wire_xf(px, py, cs.x, cs.y);
      const double* L = B.wf_line[kind][line];
      SfPt a = sf_xform_wire(m, L[0], L[1]), b = sf_xform_wire(m, L[2], L[3]);
      SfQuad q;
      if (sf_stroke_quad(a, b, q)) {
        sf_store_quad_edges(T, lane, q.p[0].x, q.p[0].y, q.p[1].x, q.p[1].y, q.p[2].x, q.p[2].y, q.p[3].x, q.p[3].y, G);
        has = G.ymin_g < G.ymax_g;
      }
    }
  }
  // bounding box of the slot's stroke: reduce over its 4 lanes
  int ymin_g = G.ymin_g, ymax_g = G.ymax_g, xmin = G.xmin, xmax = G.xmax;
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    ymin_g = min(ymin_g, __shfl_xor_sync(0xffffffffu, ymin_g, o)); ymax_g = max(ymax_g, __shfl_xor_sync(0xffffffffu, ymax_g, o));
    xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o)); xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
  }
  // one region per slot, opened in slot order by the slot's first lane
  int rid = sf_open_regions(lane, line == 0 && kind >= 0, ymin_g, ymax_g, xmin, xmax, sf_block_smem().colour_white, kind == 0 ? SF_TAG_SHIP : SF_TAG_PROJECTILE);
  rid = __shfl_sync(0xffffffffu, rid, lane & ~3);
  sf_publish_quads(W, lane, G, has, rid, line == 0 && kind >= 0, slot, kind >= 0 ? sf_block_smem().wf_nlines[kind] : 0, ymin_g, ymax_g);
  return rid;
}

// ---- ship explosion (R5 drawExplosion, draw.cpp:116-145): 84 arcs (one stroke each) + the r=7 circle -------------
// The explosion is identical for the 30 ticks a ship stays dead. On the first dead frame it is scan-converted from
// the tables of its y phase (SfExpPhase, sf_tables.h): one lane per (quad, pixel row) item adds the <= 15 tabulated
// spans of the item, shifted by the centre's x, into the item's <= SF_EXPT_NC cells (registers: nobody else adds to
// them) and tells every pixel it covers which quad did. wi / nw: this warp's index among the drawing warps.
__device__ __forceinline__ void sf_phase_exp_items(const SfDev& D, int be, int lane, int wi, int nw, int sg) {
  SfStagePool& Tm = sf_pool();
  const SfEnvRec& rec = sf_prep(sg).env[be];
  const SfPt c = sf_xform_base(rec.px, rec.py);
  const SfExpPhase& P = D.tab->exp_phase[c.y & 255];
  const int Y = c.y >> 8, bx0 = (c.x >> 8) - 13, by0 = Y - 13;  // the explosion box (sf_make_env_rec)
  const int n = __ldg(&P.n_items);
  for (int q = wi * 32 + lane; q < SF_EXP_QUADS; q += nw * 32) { Tm.exp_item0[q] = __ldg(&P.item0[q]); Tm.exp_row0[q] = __ldg(&P.row0[q]); Tm.exp_qxmin[q] = __ldg(&P.qxmin[q]); }
#pragma unroll 1
  for (int it = wi * 32 + lane; it < n; it += nw * 32) {
    const uint2 Iw = __ldg(reinterpret_cast<const uint2*>(&P.item[it]));
    const int quad = Iw.x & 255, row = Y + (int)(signed char)((Iw.x >> 8) & 255), ns = (Iw.x >> 16) & 255, span0 = Iw.y & 0xFFFF;
    const int colmin = (c.x + __ldg(&P.qxmin[quad])) >> 8;
    const int shift = c.x - (colmin << 8);
    int acc[SF_EXPT_NC];
#pragma unroll
    for (int cc = 0; cc < SF_EXPT_NC; cc++) acc[cc] = 0;
    if (row >= 0 && row < SF_NAT_H) {
      unsigned sp[SF_GRID_Y];
#pragma unroll
      for (int k = 0; k < SF_GRID_Y; k++) sp[k] = k < ns ? __ldg(reinterpret_cast<const unsigned*>(&P.span[span0 + k][0])) : 0u;
#pragma unroll
      for (int k = 0; k < SF_GRID_Y; k++) {
        const int a = (int)(short)(sp[k] & 0xFFFFu) + shift, b = (int)(short)(sp[k] >> 16) + shift;  // an unused slot has a == b
#pragma unroll
        for (int cc = 0; cc < SF_EXPT_NC; cc++) acc[cc] += max(min(b, (cc + 1) << 8) - max(a, cc << 8), 0);
      }
    }
#pragma unroll
    for (int cc = 0; cc < SF_EXPT_NC; cc++) {
      Tm.exp_len[it][cc] = (unsigned short)acc[cc];
      const int col = colmin + cc;
      if (acc[cc] && (unsigned)col < (unsigned)SF_NAT_W && (unsigned)(row - by0) < (unsigned)SF_EXP_W && (unsigned)(col - bx0) < (unsigned)SF_EXP_W) atomicOr(&Tm.arc_mask[(row - by0) * SF_EXP_W + (col - bx0)][quad >> 5], 1u << (quad & 31));
    }
  }
}

// Phase B2 (rounds that build an explosion, after sf_phase_exp_items): one lane per pixel of the 28x28 box blends
// the strokes that cover the pixel, in stroke order (arc s == quad s; the 16 chords of the circle, quads 84..99,
// are ONE stroke: their lengths add up), over the background (hexagons) and stores the sprite in the env's cache;
// the windows of phase C read it like any cached sprite. wi / nw: this warp's index among the drawing warps.
__device__ __forceinline__ void sf_phase_sprite(const SfDev& D, SfBlockSmem& B, int be, int lane, int wi, int nw, int sg) {
  SfStagePool& Tm = sf_pool();
  const SfTables* T = D.tab;
  const SfEnvRec& rec = sf_prep(sg).env[be];
  const SfPt c = sf_xform_base(rec.px, rec.py);
  const SfExpPhase& P = T->exp_phase[c.y & 255];
  const int Y = c.y >> 8, bx0 = (c.x >> 8) - 13, by0 = Y - 13;
  unsigned char* sprite = D.expc + (size_t)rec.env * (SF_EXP_W * SF_EXP_W);
#pragma unroll 1
  for (int p = wi * 32 + lane; p < SF_EXP_W * SF_EXP_W; p += nw * 32) {
    const int y = p / SF_EXP_W, x = p - y * SF_EXP_W;
    const int nx = bx0 + x, ny = by0 + y;
    unsigned v = 0;
    if ((unsigned)nx < (unsigned)SF_NAT_W && (unsigned)ny < (unsigned)SF_NAT_H) {
      v = B.bg_nat[ny * SF_NAT_STRIDE + nx];
      const uint4 M = *reinterpret_cast<const uint4*>(Tm.arc_mask[p]);
      unsigned circle = 0;
#pragma unroll 1
      for (int wd = 0; wd < 4; wd++) {
        unsigned m = wd == 0 ? M.x : wd == 1 ? M.y : wd == 2 ? M.z : M.w;
        while (m) {
          const int q = wd * 32 + __ffs(m) - 1;
          m &= m - 1;
          const int it = Tm.exp_item0[q] + (ny - Y - (int)Tm.exp_row0[q]);
          const int colmin = (c.x + Tm.exp_qxmin[q]) >> 8;
          const unsigned L = Tm.exp_len[it][nx - colmin];
          if (q < SF_EXP_STROKES - 1) v = sf_blend(v, B.exp_colour[q], sf_len_to_alpha(L));
          else circle += L;
        }
      }
      if (circle) v = sf_blend(v, B.exp_colour[SF_EXP_STROKES - 1], sf_len_to_alpha(circle));
      *reinterpret_cast<uint4*>(Tm.arc_mask[p]) = make_uint4(0u, 0u, 0u, 0u);
    }
    sprite[p] = (unsigned char)v;
  }
  if (wi == 0 && lane == 0) D.expstamp[rec.env] = rec.life;
}

// ================================================================================================================
// Block-cooperative frame pipeline. One block renders a GROUP of up to 32 envs per tick; the env records were
// written by the lanes of warp 0 (one env per lane). The strokes of all envs of the group are pooled and spread
// evenly over the warps, so that every warp of the SM runs the same phase at the same time:
//   scan   (warp 0)  strokes per env -> offsets into the round's stroke list (a round takes as many envs as fit)
//   A  env tasks     explosion sprite (first dead frame), static 16-byte output chunks, stroke list entries
//   B  stroke tasks  geometry + scan conversion of <= 8 strokes per warp into the warp's coverage cells
//   C  window tasks  one window per visible stroke / dead ship / non-zero score: composite ALL layers of the env
//                    (reading the cells of whichever warp scan-converted them) + resample + overwrite the pixels
// ================================================================================================================
struct SfFrameOut {
  unsigned char* obs;   // frames of the stage's first tick, env-major
  size_t obs_bytes;     // 84*84 or 92*90
  size_t tick_bytes;    // from one tick's frames to the next one's
  int native;           // 92x90 output (SSF_Env.step)
};
// frame of env slot e (tick e >> 5 of the stage) whose env index is `env`
__device__ __forceinline__ unsigned char* sf_frame_ptr(const SfFrameOut& out, int e, int env) {
  return out.obs + (size_t)(e >> 5) * out.tick_bytes + (size_t)env * out.obs_bytes;
}

// shells that are drawn: further than 21 from the fortress (quirk Q9, draw.cpp:249-250; sqrt-free, SfHot::touch2).
// The step computes the same mask on the fly (sf_env_step); this version is for a state that was not just stepped.
__device__ __forceinline__ unsigned sf_visible_shells(const SfDev& D, int env, unsigned pmask) {
  unsigned vis = 0;
  const double thr = D.tab->hot.touch2[2];
  for (unsigned m = (pmask >> SF_PMASK_SHELL_SHIFT) & 0xFu; m; m &= m - 1) {
    const int s = __ffs(m) - 1;
    const double2 p = D.spos[(size_t)s * D.n_pad + env];
    const double dx = SF_DSUB(p.x, SF_FORT_X), dy = SF_DSUB(p.y, SF_FORT_Y);
    if (SF_DADD(SF_DMUL(dx, dx), SF_DMUL(dy, dy)) > thr) vis |= 1u << s;
  }
  return vis;
}
// per-env stroke count (written by the env's lane before the scan)
__device__ __forceinline__ int sf_count_strokes(unsigned core, unsigned pmask, unsigned vis) {
  return ((core & SF_CORE_SHIP_ALIVE) ? 1 : 0) + __popc(pmask & SF_PMASK_MISSILES) + __popc(vis);
}

// warp 0: choose the envs of the next round (slots r_begin.. while their strokes fit) and their list offsets. The scan
// is incremental over the ticks of a stage: sf_scan_half(h) continues from the carries the previous tick left in `S`,
// sf_scan_finish publishes the round's control words; so the second tick of a stage does not scan the first one again.
struct SfScanState {
  int carry_cnt, carry_need, carry_task;
  int r1, nst, build_env, build_env2, nbuilders;
  bool closed;          // the round's last slot is known
  unsigned later_any;
};
__device__ __forceinline__ void sf_scan_begin(SfScanState& S) {
  S.carry_cnt = 0; S.carry_need = 0; S.carry_task = 0;
  S.r1 = 0; S.nst = 0; S.build_env = -1; S.build_env2 = -1; S.nbuilders = 0;
  S.closed = false; S.later_any = 0u;
}
// slots 32h .. 32h + 31 (tick h of the stage); r_begin: first slot that still has to be drawn
__device__ __forceinline__ void sf_scan_half(SfStagePrep& Tm, int lane, int h, int r_begin, SfScanState& S) {
  if (!S.closed) S.r1 = 32 * (h + 1);
  const int slot = 32 * h + lane;
  SfEnvRec& rec = Tm.env[slot];
  const bool cand = slot >= r_begin && rec.env >= 0;
  const int cnt = cand ? rec.ns : 0;
  int need = 0;  // worst-case coverage cells of this env's regions
  if (cand) need = ((rec.core & SF_CORE_SHIP_ALIVE) ? SF_CELLS_SHIP : 0) + __popc(rec.pmask & SF_PMASK_MISSILES) * SF_CELLS_MISSILE + __popc(rec.shell_vis) * SF_CELLS_SHELL;
  // window tasks of the round that do not belong to a stroke: the stale quarters of a dead ship's explosion box,
  // the strip of a non-zero score (the static base shows "0000000")
  const bool deadc = cand && !(rec.core & SF_CORE_SHIP_ALIVE), scorec = cand && rec.points_i > 0;
  const int qvalidc = deadc ? (rec.building >> 4) & 15 : 0;
  const int cnttc = (deadc ? 4 - __popc(qvalidc) : 0) + (scorec ? 1 : 0);
  // one scan for the three counters: strokes (8 bits per env are not enough for the sum: 10 bits), cells (15 bits), tasks (9 bits)
  unsigned long long packed = (unsigned long long)cnt | ((unsigned long long)need << 12) | ((unsigned long long)cnttc << 32);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, packed, o); if (lane >= o) packed += t; }
  const int incl = (int)(packed & 0xFFFu) + S.carry_cnt, incl_need = (int)((packed >> 12) & 0xFFFFFu) + S.carry_need;
  const int inclt_all = (int)(packed >> 32);
  const unsigned builders = __ballot_sync(0xffffffffu, cand && (rec.building & 1));
  // a round builds the explosions of at most two envs: the round ends before the third builder
  unsigned third = builders;
  for (int k = S.nbuilders; k < 2 && third; k++) third &= third - 1;
  const unsigned over = __ballot_sync(0xffffffffu, incl > SF_ROUND_STROKES || incl_need > SF_POOL_CELLS) | (third ? ~((third & (0u - third)) - 1u) : 0u);
  if (!S.closed && over) { S.r1 = 32 * h + __ffs(over) - 1; S.closed = true; }
  for (unsigned bm = builders; bm && S.build_env2 < 0; bm &= bm - 1) {
    const int sl = 32 * h + __ffs(bm) - 1;
    if (S.build_env < 0) S.build_env = sl; else S.build_env2 = sl;
  }
  S.nbuilders += __popc(builders);
  const bool in_round = cand && slot < S.r1;
  if (in_round) rec.s0 = incl - cnt;
  // strokes of the round = inclusive count of its last slot
  const unsigned inr = __ballot_sync(0xffffffffu, in_round);
  if (inr) S.nst = __shfl_sync(0xffffffffu, incl, 31 - __clz((int)inr));
  S.later_any |= __ballot_sync(0xffffffffu, cand && slot >= S.r1);
  // tasks are counted for the slots IN the round only: the slots of a half that are in the round are a prefix of the half,
  // so the inclusive task count of the round's last slot of this half is what carries over
  if (in_round) {
    int k = inclt_all - cnttc + S.carry_task;
    if (deadc) for (int q = 0; q < 4; q++) if (!((qvalidc >> q) & 1)) Tm.etask[k++] = (unsigned short)(slot | (q << 6));
    if (scorec) Tm.etask[k] = (unsigned short)(slot | (4 << 6));
  }
  if (inr) S.carry_task += __shfl_sync(0xffffffffu, inclt_all, 31 - __clz((int)inr));
  S.carry_cnt = __shfl_sync(0xffffffffu, incl, 31); S.carry_need = __shfl_sync(0xffffffffu, incl_need, 31);
}
__device__ __forceinline__ void sf_scan_finish(SfStagePrep& Tm, int lane, int r_begin, const SfScanState& S) {
  if (lane == 0) {
    Tm.more = S.later_any != 0u;
    Tm.r0 = r_begin; Tm.r1 = S.r1; Tm.nstrokes = S.nst;
    Tm.build_env = (S.build_env >= 0 && S.build_env < S.r1) ? S.build_env : -1;
    Tm.build_env2 = (Tm.build_env >= 0 && S.build_env2 >= 0 && S.build_env2 < S.r1) ? S.build_env2 : -1;
    // phase B1 hands the strokes out in equal batches of <= 8, one per drawing warp
    // (the last drawing warps get no batch: one of them issues the round's bulk copies instead, see sf_draw_stage)
    Tm.chunk = min(max((S.nst + SF_CHUNK_WARPS - 1) / SF_CHUNK_WARPS, 1), 8);
    Tm.netask = S.carry_task;
  }
  __syncwarp();
}
// the whole scan at once (a later round of a stage: slots r_begin .. nslots - 1)
__device__ __forceinline__ void sf_round_scan(SfStagePrep& Tm, int lane, int r_begin, int nslots) {
  SfScanState S;
  sf_scan_begin(S);
#pragma unroll
  for (int h = 0; h < SF_STAGE_TICKS; h++)
    if (32 * h < nslots && 32 * (h + 1) > r_begin) sf_scan_half(Tm, lane, h, r_begin, S);
  sf_scan_finish(Tm, lane, r_begin, S);
}

// Static base of the observation of env slot e: the whole default observation (hexagons, "0000000", empty bar) goes
// out as ONE asynchronous bulk copy from the block's shared-memory copy (TMA engine, 7056 bytes; one copy per lane of
// the issuing warp, see sf_draw_stage)...
__device__ __forceinline__ void sf_env_base_issue(const SfBlockSmem& B, int e, const SfFrameOut& out, int sg) {
  const int env = sf_prep(sg).env[e].env;
  if (env < 0) return;
  const unsigned src = (unsigned)__cvta_generic_to_shared(B.bg_obs);
  unsigned char* gb = sf_frame_ptr(out, e, env);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gb), "r"(src), "r"(84 * 84) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// ... and, once the bulk copies have landed, the few 16-byte chunks that the fortress state (about 12
// for a live fortress, 53 for its explosion) and a non-empty vulnerability bar change are patched from the
// pre-resampled state tables.
__device__ __forceinline__ void sf_env_base_patch(const SfDev& D, const SfBlockSmem& B, int lane, int e, const SfFrameOut& out, int sg) {
  const SfTables* T = D.tab;
  const SfEnvRec& rec = sf_prep(sg).env[e];
  const int env = rec.env;
  if (env < 0) return;
  const unsigned core = rec.core;
  const int fst = (core & SF_CORE_FORT_ALIVE) ? (int)((core >> SF_CORE_FANG_SHIFT) & 63u) : 36;
  const int bst = rec.kill_bar ? 11 : min(rec.vuln, 10);
  int4* g = reinterpret_cast<int4*>(sf_frame_ptr(out, e, env));
  const int4* ft = reinterpret_cast<const int4*>(T->obs_fort[fst]);
  const int fc0 = T->fort_chunk0;
  // lanes 0..15: fortress chunks (index list in shared memory), lanes 0..20: bar chunks; both loads in flight
  const int c0 = lane < 16 ? B.fort_sparse[fst][lane] : 255;
  const bool bar = bst != 0 && lane < SF_OBS_CHUNKS - SF_BAR_CHUNK0;
  int4 v0, vb;
  if (c0 != 255) v0 = __ldg(&ft[c0]);
  if (bar) vb = __ldg(reinterpret_cast<const int4*>(T->obs_bar[bst]) + lane);
  if (c0 != 255) g[fc0 + c0] = v0;
  if (bar) g[SF_BAR_CHUNK0 + lane] = vb;
  if (fst == 36) {  // fortress explosion: the rest of its 53 chunks
    const int nsp = T->fort_sparse_n[fst];
#pragma unroll 1
    for (int k = 16 + lane; k < nsp; k += 32) { const int c = T->fort_sparse[fst][k]; g[fc0 + c] = __ldg(&ft[c]); }
  }
  // dead ship: the quarters of its resampled explosion box that are still valid are copied, not recomputed (a
  // wireframe that reaches into the box gets its own window in phase C, which composites the explosion under it)
  const int qvalid = !(core & SF_CORE_SHIP_ALIVE) ? (rec.building >> 4) & 15 : 0;
  if (qvalid) {
    __syncwarp();  // the chunk stores above and the byte stores below (other lanes) can touch the same bytes: order them
    const int bx0 = (rec.ebox & 255) - 64, by0 = ((rec.ebox >> 8) & 255) - 64;
    const int x0 = max(bx0, 0), y0 = max(by0, 0), x1 = min(bx0 + SF_EXP_W, SF_NAT_W) - 1, y1 = min(by0 + SF_EXP_W, SF_NAT_H) - 1;
    if (x0 <= x1 && y0 <= y1) {
      const int j0 = B.col_out0[x0], j1 = B.col_out1[x1], i0 = B.row_out0[y0], i1 = B.row_out1[y1];
      const int hb = (i1 - i0 + 4) >> 2, oh = i1 - i0 + 1;
      const int ja = j0 & ~3;  // the cache columns start at a 32-bit word of the observation row (rows are 84 = 4 * 21 bytes)
      const unsigned* src = reinterpret_cast<const unsigned*>(D.expo + (size_t)env * SF_EXPO_BYTES);
      unsigned char* dst = sf_frame_ptr(out, e, env) + i0 * 84 + ja;
      // valid rows as a bit mask (row r belongs to quarter r / hb)
      unsigned rows = 0u;
#pragma unroll
      for (int q = 0; q < 4; q++)
        if ((qvalid >> q) & 1) { const int ra = q * hb, rb = min(ra + hb, oh); if (ra < rb) rows |= ((rb - ra >= 32 ? 0u : (1u << (rb - ra))) - 1u) << ra; }
      const int wfull0 = (j0 - ja + 3) >> 2, wfull1 = (j1 + 1 - ja) >> 2;  // words [wfull0, wfull1) lie inside [j0, j1]
      // whole words: 8 per row
      unsigned v[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int k = lane + 32 * u, w = k & 7;
        const bool on = ((rows >> (k >> 3)) & 1u) && w >= wfull0 && w < wfull1;
        v[u] = on ? __ldcg(&src[k]) : 0u;
      }
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int k = lane + 32 * u, w = k & 7;
        if (((rows >> (k >> 3)) & 1u) && w >= wfull0 && w < wfull1) *reinterpret_cast<unsigned*>(dst + (k >> 3) * 84 + 4 * w) = v[u];
      }
      // the (at most two) partial words at the ends of a row: lane = row
      if ((rows >> lane) & 1u) {
        const int wl = wfull0 - 1, wr = wfull1;   // partial iff they hold a column of [j0, j1]
        if (wl >= 0) {
          const unsigned x = __ldcg(&src[lane * 8 + wl]);
          unsigned char* p = dst + lane * 84 + 4 * wl;
#pragma unroll
          for (int b = 0; b < 4; b++) { const int c = ja + 4 * wl + b; if (c >= j0 && c <= j1) p[b] = (unsigned char)(x >> (8 * b)); }
        }
        if (wr != wl && ja + 4 * wr <= j1) {
          const unsigned x = __ldcg(&src[lane * 8 + wr]);
          unsigned char* p = dst + lane * 84 + 4 * wr;
#pragma unroll
          for (int b = 0; b < 4; b++) { const int c = ja + 4 * wr + b; if (c >= j0 && c <= j1) p[b] = (unsigned char)(x >> (8 * b)); }
        }
      }
    }
  }
}

// Stepping warp, after the round scan of the stage it prepares: the strokes of the round's slots of tick `h` of the
// stage, one env per lane, from the SoA state (which holds exactly that tick): [ship] + live missiles (slot order) +
// visible shells (slot order) == draw order.
__device__ __forceinline__ void sf_gather_strokes(const SfDev& D, SfStagePrep& Tm, int lane, int h) {
  const int slot = 32 * h + lane;
  const SfEnvRec& rec = Tm.env[slot];
  if (slot >= Tm.r0 && slot < Tm.r1 && rec.env >= 0) {
    const int env = rec.env, np = D.n_pad;
    const unsigned core = rec.core;
    SfStrokeRec* S = &Tm.stroke[rec.s0];
    if (core & SF_CORE_SHIP_ALIVE) { S->x = rec.px; S->y = rec.py; S->desc = 0 | ((int)(core & SF_CORE_ANGLE_MASK) << 2) | (slot << 12); S++; }
    // (up to three missiles per trip: the loads of a trip are in flight together — each is an L2 round trip for this one
    // warp. Plain scalars: indexed arrays end up in local memory here)
    for (unsigned m = rec.pmask & SF_PMASK_MISSILES; m;) {
      const int k0 = __ffs(m) - 1; m &= m - 1;
      const int k1 = m ? __ffs(m) - 1 : k0; m &= m - 1;
      const int k2 = m ? __ffs(m) - 1 : k0; m &= m - 1;
      const double2 p0 = D.mpos[(size_t)k0 * np + env], p1 = D.mpos[(size_t)k1 * np + env], p2 = D.mpos[(size_t)k2 * np + env];
      const int a0 = D.mang[(size_t)k0 * np + env], a1 = D.mang[(size_t)k1 * np + env], a2 = D.mang[(size_t)k2 * np + env];
      S->x = p0.x; S->y = p0.y; S->desc = 1 | (a0 << 2) | (slot << 12); S++;
      if (k1 != k0) { S->x = p1.x; S->y = p1.y; S->desc = 1 | (a1 << 2) | (slot << 12); S++; }
      if (k2 != k0) { S->x = p2.x; S->y = p2.y; S->desc = 1 | (a2 << 2) | (slot << 12); S++; }
    }
    for (unsigned m = (unsigned)rec.shell_vis; m; m &= m - 1) {
      const int k = __ffs(m) - 1;
      const double2 p = D.spos[(size_t)k * np + env];
      int angle = __double2int_rz(D.sang[(size_t)k * np + env]);  // `int angle` truncation, quirk Q10
      if (angle >= 360) angle -= 360;
      S->x = p.x; S->y = p.y; S->desc = 2 | (angle << 2) | (slot << 12); S++;
    }
  }
  __syncwarp();
}

// phase B for this warp. B1: warp wi builds the geometry of batch wi (Tm.chunk consecutive strokes of the round's
// list: at most one batch per warp) and publishes its records; after a barrier of the drawing warps, B3: the
// passes of ALL batches are dealt round-robin over ALL drawing warps, so the scan conversion is balanced whatever
// the size of the individual strokes.
__device__ __forceinline__ void sf_phase_strokes(const SfDev& D, SfBlockSmem& B, SfWarpSmem& W, int lane, int wi, int nw, int nst, int sg) {
  const SfTables* T = D.tab;
  const SfStagePrep& Tm = sf_prep(sg);
  const int chunk = Tm.chunk;
  // B2, first half: the items of the explosion of a ship that died in this stage. They are dealt from the LAST
  // drawing warp down: the geometry batches go to the first warps, so the two overlap.
  const int be = Tm.build_env;
  if (be >= 0) sf_phase_exp_items(D, be, lane, nw - 1 - wi, nw, sg);
  const int s = wi * chunk;
  if (s < nst) {
    const int slot = lane >> 2;
    const bool valid = slot < chunk && s + slot < nst;
    const int idx = s + slot;
    int kind = -1, angle = 0;
    double x = 0, y = 0;
    if (valid) {
      const SfStrokeRec& S = Tm.stroke[idx];
      x = S.x; y = S.y; kind = S.desc & 3; angle = (S.desc >> 2) & 1023;
    }
    const int rid = sf_wire_geometry(W, lane, T, kind, x, y, angle);
    if (valid && (lane & 3) == 0) sf_pool().stroke_region[idx] = (short)rid;
  } else {
    if (lane == 0) W.ngroups = 0;
  }
  sf_render_sync();  // every batch is published, the explosion items are done
  // B2, second half: the sprite (its stamp is visible to the stepping warp long before it looks at the next stage). A
  // round takes at most two explosions; they share the item lengths and the pixel masks, one after the other.
  if (be >= 0) {
    sf_phase_sprite(D, B, be, lane, wi, nw, sg);
    if (Tm.build_env2 >= 0) {
      sf_render_sync();
      sf_phase_exp_items(D, Tm.build_env2, lane, wi, nw, sg);
      sf_render_sync();
      sf_phase_sprite(D, B, Tm.build_env2, lane, wi, nw, sg);
    }
  }
  // passes of warp l's batch: (ngroups + 3) / 4; every warp computes the same prefix sums
  const int mine = lane < nw ? (sf_warp_smem(lane + 1).ngroups + 3) >> 2 : 0;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
#pragma unroll 1
  for (int g = wi; g < total; g += nw) {
    const int owner = __popc(__ballot_sync(0xffffffffu, incl <= g));  // first warp whose inclusive count exceeds g
    const int first = __shfl_sync(0xffffffffu, incl - mine, owner);
    sf_accumulate_pass(owner + 1, (g - first) << 2);
  }
}

// phase C task t of this round: env tasks (quarters of explosion boxes, score strips) first, then one per stroke
__device__ __forceinline__ void sf_phase_window(const SfDev& D, SfBlockSmem& B, SfWarpSmem& W, int lane, int t, int netask, const SfFrameOut& out, int sg) {
  const SfTables* T = D.tab;
  int e, j0, i0, j1, i1;
  int quarter = -1, corigin = 0;
  if (t < netask) {
    const int et = sf_prep(sg).etask[t], kind = et >> 6;
    e = et & 63;
    const SfEnvRec& rec = sf_prep(sg).env[e];
    int x0, y0, x1, y1;
    if (kind < 4) {  // dead ship: a quarter (in output rows) of the explosion box
      const int bx0 = (rec.ebox & 255) - 64, by0 = ((rec.ebox >> 8) & 255) - 64;
      x0 = max(bx0, 0); y0 = max(by0, 0); x1 = min(bx0 + SF_EXP_W, SF_NAT_W) - 1; y1 = min(by0 + SF_EXP_W, SF_NAT_H) - 1;
      if (x0 > x1 || y0 > y1) return;
    } else {         // non-zero score: the static base shows "0000000"
      x0 = SF_TEXT_X0; y0 = SF_TEXT_Y0; x1 = SF_TEXT_X0 + SF_TEXT_W - 1; y1 = SF_TEXT_Y0 + SF_TEXT_H - 1;
    }
    j0 = B.col_out0[x0]; j1 = B.col_out1[x1]; i0 = B.row_out0[y0]; i1 = B.row_out1[y1];
    if (kind < 4) {
      const int hb = (i1 - i0 + 4) >> 2;
      corigin = (j0 & ~3) | (i0 << 8);  // cache columns are aligned with the 32-bit words of the observation row
      i0 += kind * hb; i1 = min(i1, i0 + hb - 1);
      if (i0 > i1) return;
      quarter = (rec.building & 2) ? kind : -1;  // may this round refresh the env's cache (sf_publish_recs)?
    }
  } else {
    const int sr = sf_pool().stroke_region[t - netask];
    if (sr < 0) return;
    e = sf_prep(sg).stroke[t - netask].desc >> 12;
    const int4 R = sf_pool().region[sr];
    j0 = B.col_out0[R.x]; j1 = B.col_out1[R.x + (R.z & 0xFFFF) - 1]; i0 = B.row_out0[R.y]; i1 = B.row_out1[R.y + ((R.z >> 16) & 0xFFFF) - 1];
  }
  const int env = sf_prep(sg).env[e].env;
  const bool cached = sf_window_orect(T, D.expc + (size_t)env * (SF_EXP_W * SF_EXP_W), e, j0, i0, j1, i1, sf_frame_ptr(out, e, env),
                                      quarter >= 0 ? D.expo + (size_t)env * SF_EXPO_BYTES : nullptr, corigin, sg);
  if (cached && lane == 0) {
    // mark the quarter valid, unless the stepping warp has already re-keyed the cache for the next tick
    const SfEnvRec& rec = sf_prep(sg).env[e];
    const unsigned long long want = (unsigned long long)rec.life | ((unsigned long long)sf_expo_key(rec) << 32);
    unsigned long long* m = reinterpret_cast<unsigned long long*>(&D.expo_meta[env]);
    unsigned long long old = *reinterpret_cast<volatile unsigned long long*>(m);
    while ((old & 0x0FFFFFFFFFFFFFFFull) == want) {
      const unsigned long long prev = atomicCAS(m, old, old | (1ull << (60 + quarter)));
      if (prev == old) break;
      old = prev;
    }
  }
  (void)W;
}

// native output (SSF_Env.step returns the 92x90 frame): tile `tile` (30x30 windows, 3 x 4 of them) of env slot e
__device__ __forceinline__ void sf_phase_native_tile(const SfDev& D, SfBlockSmem& B, SfWarpSmem& W, int lane, int e, int tile, const SfFrameOut& out, int sg) {
  const int env = sf_prep(sg).env[e].env;
  if (env < 0) return;
  const int tx = (tile % 3) * 30, ty = (tile / 3) * 30;
  const int pw = min(30, SF_NAT_W - tx), ph = min(30, SF_NAT_H - ty);
  const int win = tx | (ty << 8) | (pw << 16) | (ph << 24);
  (void)sf_composite(D.tab, D.expc + (size_t)env * (SF_EXP_W * SF_EXP_W), e, win, sg);
  unsigned char* dst = sf_frame_ptr(out, e, env) + ty * SF_NAT_W + tx;
  sf_for_rect(lane, pw, ph, [&](int c, int r) { dst[r * SF_NAT_W + c] = W.patch[r * SF_PATCH_STRIDE + c]; });
  __syncwarp();
}

// warp 0, one env per lane, on the records of tick h of the stage being prepared in ring slot `cur`: a dead ship whose
// explosion sprite is neither cached nor built by an earlier round gets it built in this round (bit 0); which quarters
// of its resampled explosion box are valid (bits 4..7) and whether this round may refresh them (bit 1).
// The stages still in the ring (the other slots, and the earlier tick of this one) were prepared before this one and
// may not have been drawn yet; everything older has (warp 0 waited for the slot it now fills). Stages are drawn in the
// order they were prepared, and a stage's writes to the caches are complete before the next one starts.
//  * Sprite (expc / expstamp; written only by the build of (env, life)). A stamp equal to the life means the build has
//    been drawn. An earlier record of the same env and life in the ring means that stage builds the sprite, or found it
//    cached or scheduled itself: either way it exists before this stage is drawn, so it is not built again (with two
//    stages of lead a death would otherwise be built three times; the round scan takes two builds per round). Nothing
//    overwrites it in between: an earlier undrawn stage builds only for a life it holds, and a different life of the same
//    env earlier in time would put this life's death (and its first build) after that stage.
//  * Resampled box (expo / expo_meta). Warp 0 re-keys the meta, in preparation order, to (life, key) whenever a record
//    differs from it; a window sets a quarter's valid bit with a compare-and-swap against its own (life, key), so bits are
//    only ever set on the key they were computed for, and a stage trusts the bits it finds on its own key. The hazard of
//    a lead: a window of an earlier, still undrawn stage with ANOTHER key overwriting the bytes of a quarter whose bit a
//    stage of this key has set (or will set) after the re-key. So a stage may write the cache only if no record of the
//    env in the ring has another (life, key) (bit 1). Then the last write of a quarter before a stage X that trusts it
//    came from a stage W of X's key: a W with another key prepared after the re-key R would have re-keyed again, and one
//    prepared before R was drawn after the stage Z of X's key that set the bit, so Z was undrawn and in the ring when W
//    was prepared, which denies W the write. This costs the cache only the stages around a key change. The valid bits a
//    stage finds are those of the stages drawn SF_PREP_SLOTS - 1 before it or earlier (one more stage of lag than with
//    one stage of lead); the refreshes in between recompute identical pixels.
__device__ __forceinline__ void sf_publish_recs(const SfDev& D, SfStagePrep* ring, int cur, int lane, int h, bool native) {
  SfEnvRec& r = ring[cur].env[32 * h + lane];
  if (r.env >= 0 && !(r.core & SF_CORE_SHIP_ALIVE)) {
    const unsigned stamp = __ldcg(&D.expstamp[r.env]);  // both loads in flight together
    const unsigned long long mw = __ldcg(reinterpret_cast<const unsigned long long*>(&D.expo_meta[r.env]));
    const unsigned mx = (unsigned)mw, my = (unsigned)(mw >> 32);
    const unsigned key = sf_expo_key(r);
    int building = stamp != r.life ? 1 : 0;
    bool refresh = true;
#pragma unroll 1
    for (int k = 0; k < SF_PREP_SLOTS * SF_STAGE_TICKS; k++) {
      const int j = k / SF_STAGE_TICKS, hh = k - j * SF_STAGE_TICKS;
      if (j == cur && hh >= h) continue;
      const SfEnvRec& o = ring[j].env[32 * hh + lane];
      if (o.env != r.env || (o.core & SF_CORE_SHIP_ALIVE)) continue;
      if (o.life == r.life) building = 0;
      if (o.life != r.life || sf_expo_key(o) != key) refresh = false;
    }
    if (!native) {
      const bool same = mx == r.life && (my & 0x0FFFFFFFu) == key;
      if (same) { if (!building) building |= (int)(my >> 28) << 4; }
      else atomicExch(reinterpret_cast<unsigned long long*>(&D.expo_meta[r.env]), (unsigned long long)r.life | ((unsigned long long)key << 32));
    }
    r.building = building | (refresh ? 2 : 0);
  }
  __syncwarp();
}

// what persists from one group of envs to the next in a persistent block
struct SfStageState {
  int stage;      // ring slot the next stage is drawn from
  int prev_used;  // coverage cells the previous stage used: zeroed at the start of the next one
};

// warp 0: the first round of a new stage in ring slot sg: up to SF_STAGE_TICKS consecutive ticks starting at tick t (nt
// of them are left). prep(t, Tm, h) writes the env records of tick t into slots 32h .. 32h + 31 and leaves the SoA state
// at that tick. The strokes of a tick are gathered from the state before it moves on, so the first tick must fit the
// round in one piece; if it does not, the stage covers that tick only (and takes several rounds).
template <class Prep>
__device__ __forceinline__ void sf_prepare_first_round(const SfDev& D, SfBlockSmem& B, int sg, int lane, int t, int nt, SfFrameOut out, Prep prep) {
  SfStagePrep& Tm = B.prep[sg];
  const bool native = out.native != 0;
  SF_BT_BEGIN();
  prep(t, Tm, 0);
  SF_BT(3);
  sf_publish_recs(D, B.prep, sg, lane, 0, native);
  SF_BT(4);
  SfScanState S;
  sf_scan_begin(S);
  sf_scan_half(Tm, lane, 0, 0, S);
  sf_scan_finish(Tm, lane, 0, S);
  SF_BT(5);
  sf_gather_strokes(D, Tm, lane, 0);
  SF_BT(6);
  int nticks = 1;
  if (nt > 1 && !Tm.more) {
    prep(t + 1, Tm, 1);
    SF_BT(3);
    sf_publish_recs(D, B.prep, sg, lane, 1, native);
    SF_BT(4);
    sf_scan_half(Tm, lane, 1, 0, S);   // continues the first tick's scan (the round was not closed: !Tm.more)
    sf_scan_finish(Tm, lane, 0, S);
    SF_BT(5);
    sf_gather_strokes(D, Tm, lane, 1);
    SF_BT(6);
    nticks = 2;
  }
  if (lane == 0) Tm.nticks = nticks;
  __syncwarp();
  SF_BT(7);
}

// One stage drawn by the 23 drawing warps (see the pipeline description above): B1 geometry, B3 passes, base
// patches, B2 explosion sprite, C windows. Returns the coverage cells the stage used (zeroed at the start of the next).
__device__ __forceinline__ int sf_draw_stage(const SfDev& D, SfBlockSmem& B, SfWarpSmem& W, int lane, const SfFrameOut& out, int sg) {
  const int warp = threadIdx.x >> 5;
  const int wi = warp - 1, nw = SF_RENDER_WARPS - 1;  // index among the drawing warps, and their number
  const SfStagePrep& Tm = B.prep[sg];
  SfStagePool& P = B.pool;
  const int r0 = Tm.r0, r1 = Tm.r1, nst = Tm.nstrokes;
  // ---- B: stroke tasks ----
  // The default observations of the round go out as bulk copies issued by ONE warp, the last drawing warp, one copy per
  // lane: it has no geometry batch (Tm.chunk), so the time the copy engine's queue makes an issuer wait (when all 23 warps
  // issued their two or three copies at the same moment that was 7 % of all stall samples) is spent by a warp that would
  // idle; after its share of the passes it waits for the copies (long done) and raises Tm.base_ready, which the other warps
  // look at before they patch.
  const bool base_issuer = !out.native && wi == nw - 1;
  if (base_issuer) {
#pragma unroll 1
    for (int e = r0 + lane; e < r1; e += 32) sf_env_base_issue(B, e, out, sg);
  }
  sf_phase_strokes(D, B, W, lane, wi, nw, nst, sg);
  if (!out.native) {
    // the copies were issued a whole phase ago: the issuer's wait returns at once, and so does everybody's look at the flag
    if (base_issuer) {
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      __syncwarp();
      if (lane == 0) { __threadfence_block(); *(volatile int*)&P.base_ready = 1; }
    } else {
      while (*(volatile int*)&P.base_ready == 0) {}
    }
    __syncwarp();
    // first come first served: the warps leave the passes one pass apart, and a patch is as long as a pass
#pragma unroll 1
    for (;;) {
      int e = 0;
      if (lane == 0) e = atomicAdd(&P.next_patch, 1);
      e = r0 + __shfl_sync(0xffffffffu, e, 0);
      if (e >= r1) break;
      sf_env_base_patch(D, B, lane, e, out, sg);
    }
  }
  const int used = P.cells_used;  // final since the geometry barrier in sf_phase_strokes
  sf_render_sync();
  // the counters of B are not touched again in this stage: restart them for the next one (its B1 starts after every
  // drawing warp has synced on the next stage's full barrier)
  if (threadIdx.x == 32) { P.nregions = 0; P.cells_used = 0; P.next_patch = 0; P.base_ready = 0; }
  // ---- C: window tasks, handed out first come first served (env tasks first: the big ones) ----
  if (!out.native) {
    const int netask = Tm.netask;
#pragma unroll 1
    for (;;) {
      int t = 0;
      if (lane == 0) t = atomicAdd(&P.next_task, 1);
      t = __shfl_sync(0xffffffffu, t, 0);
      if (t >= netask + nst) break;
      sf_phase_window(D, B, W, lane, t, netask, out, sg);
    }
  } else {
#pragma unroll 1
    for (int t = wi; t < (r1 - r0) * 12; t += nw) sf_phase_native_tile(D, B, W, lane, r0 + t / 12, t % 12, out, sg);
  }
  return used;
}

// All frames of T consecutive ticks of one group, as two ROLES that run the same stage sequence: sf_stepper_ticks
// (warp 0) and sf_drawer_ticks (the other warps). prep(t, Tm, h) is executed by warp 0 only and writes the env records
// of tick t into Tm.env[32h ..] (one env per lane, env = -1: unused); for a rollout it is the step of tick t, which
// therefore runs while the other warps draw the ticks before it.
// A STAGE is a round of up to SF_STAGE_TICKS consecutive ticks, prepared in ring slot s % SF_PREP_SLOTS. Warp 0 fills
// the slots in drawing order and hands each one over at its full barrier; it waits (empty barrier) only when it is
// SF_PREP_SLOTS stages ahead of the drawing warps, so a slow stage on one side is absorbed by the lead instead of
// stalling the other side. Nothing of a stage that is being drawn reads the SoA state, so the steps may overwrite it;
// the strokes of a LATER round of the same stage are gathered (from the state, which still holds the stage's last tick)
// before the next step.
// The roles are separate functions on purpose: the rollout kernel calls them out of line, so that each role gets its own
// register allocation (sharing one loop, the long-lived variables of the drawing warps were spilled around the stepping
// warp's calls and reloaded inside the drawing code: nvdisasm -g attribution of LDL / STL).

// warp 0: the ring slot of its stage number `stage` (stages prepared by the block so far), once the drawing warps have
// drawn what the slot held
__device__ __forceinline__ int sf_stepper_claim(int stage) {
  const int sg = stage % SF_PREP_SLOTS;
  SF_TL(4);
  if (stage >= SF_PREP_SLOTS) sf_stage_empty_wait(sg);
  SF_TL(5);
  return sg;
}
// warp 0, at the end of the kernel: take the drawing warps' arrivals for the last stages, so that no named barrier is
// left half arrived
__device__ __forceinline__ void sf_stepper_drain(int stage) {
#pragma unroll 1
  for (int s = max(stage - SF_PREP_SLOTS, 0); s < stage; s++)
    asm volatile("bar.sync %0, %1;" :: "r"(3 + SF_PREP_SLOTS + s % SF_PREP_SLOTS), "r"(32 * SF_RENDER_WARPS) : "memory");
}

template <class Prep>
__device__ __forceinline__ void sf_stepper_ticks(const SfDev& D, SfBlockSmem& B, int lane, bool native, int T, int& stage, Prep prep) {
  SfFrameOut out;
  out.obs = nullptr; out.obs_bytes = 0; out.tick_bytes = 0; out.native = native ? 1 : 0;
  int sg = sf_stepper_claim(stage);
  sf_prepare_first_round(D, B, sg, lane, 0, T, out, prep);
  SF_TL(3);
  int t = 0;
#pragma unroll 1
  for (;;) {
    sf_stage_full_arrive(sg);  // the stage is prepared
    stage++;
    const SfStagePrep& Tm = B.prep[sg];
    const bool more = Tm.more != 0;            // more env slots in the stage than this round could take?
    const int nticks = Tm.nticks;
    if (!more && t + nticks >= T) break;
    const int nx = sf_stepper_claim(stage);
    SfStagePrep& Nx = B.prep[nx];
    if (more) {
#pragma unroll
      for (int h = 0; h < SF_STAGE_TICKS; h++) Nx.env[32 * h + lane] = Tm.env[32 * h + lane];
      if (lane == 0) Nx.nticks = nticks;
      __syncwarp();
      sf_round_scan(Nx, lane, Tm.r1, SF_GROUP_ENVS * nticks);
      sf_gather_strokes(D, Nx, lane, nticks - 1);  // the slots that are left are of the stage's last tick (see above)
    } else {
      sf_prepare_first_round(D, B, nx, lane, t + nticks, T - (t + nticks), out, prep);
      t += nticks;
    }
    sg = nx;
  }
  SF_TL(7);
}

__device__ __forceinline__ void sf_drawer_ticks(const SfDev& D, SfBlockSmem& B, SfWarpSmem& W, int lane, SfFrameOut out, int T, SfStageState& st) {
  unsigned char* const obs0 = out.obs;
  int t = 0;
#pragma unroll 1
  for (;;) {
    const int sg = st.stage;
    SF_TL(4);
    sf_stage_full_wait(sg);  // the stage is prepared, and every drawing warp is done with the one before it
    SF_TL(5);
    const SfStagePrep& Tm = B.prep[sg];
    const bool more = Tm.more != 0;
    const int nticks = Tm.nticks;
    const bool last = !more && t + nticks >= T;
    // the pool is the previous stage's until here: zero the coverage cells it used (before the passes of this stage,
    // which follow the geometry barrier) and restart the window queue (used after the second barrier)
    {
      const int nz = (st.prev_used + 1) >> 1;
      for (int k = threadIdx.x - 32; k < nz; k += 32 * (SF_RENDER_WARPS - 1)) reinterpret_cast<unsigned*>(B.pool.cells)[k] = 0u;
      if (threadIdx.x == 32) B.pool.next_task = 0;
    }
    out.obs = obs0 + (size_t)t * out.tick_bytes;
    st.prev_used = sf_draw_stage(D, B, W, lane, out, sg);
    sf_stage_empty_arrive(sg);  // the slot may be refilled
    st.stage = sg + 1 == SF_PREP_SLOTS ? 0 : sg + 1;
    if (!more) t += nticks;
    if (last) break;
  }
  SF_TL(7);
}
