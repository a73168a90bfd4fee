/* tbx_render.cuh -- the canvas render kernel (Toybox.get_state / get_rgb_frame), and the draw-list helpers the other
 * renderers share.
 *
 * The native layouts (RGBA / RGB / gray) are rendered as broadcast + patch (tbx_render_native.cuh).  Breakout and
 * Amidar envs that differ from their base frame in many places are handed to this kernel instead.
 *
 * DELTA RENDERING over a persistent shared-memory canvas.  One CTA owns a band of canvas rows and renders it for a
 * chunk of TBX_EPC = 8 consecutive envs (8 envs x 4 B = one 32-byte sector per state word, so the word-major
 * planes are read at full sector efficiency).
 *   - The canvas is initialised ONCE per CTA from a pre-rendered BASE FRAME of the pool's config (base 0: static
 *     draw-list slots -- walls, ground line; base 1: plus the look of a fresh game -- all bricks / the config's
 *     tile board), kept in L2.
 *   - Per env only the draw-list entries that differ from the base are built (straight from the env's record)
 *     and painted, group by group in draw order.  Inside a group whose primitives cannot conflict (disjoint, or
 *     one colour) every thread paints its own small rectangle with 32-bit span stores, larger / sprite-masked
 *     primitives are painted warp-cooperatively; groups that may conflict are painted by one warp strictly in
 *     order.  The result equals the painter's algorithm over the full draw list.  Painted areas are recorded as
 *     dirty rectangles.
 *   - The painted band leaves for the destination frame through the TMA engine.
 *   - Afterwards the dirty rectangles are restored from the base frame, so per-env work is proportional to what
 *     differs from the base, not to the frame size.
 */
#ifndef TBX_RENDER_CUH
#define TBX_RENDER_CUH
#include <cuda_runtime.h>
#include "tbx_breakout.h"
#include "tbx_space_invaders.h"
#include "tbx_amidar.h"

namespace tbxk {

/* The kernel is compiled for up to 256 threads and 64 registers per thread (4 x 256 or 8 x 128 threads per SM);
 * the launch picks the CTA size per game.  The CTA size is a power of two. */
#define TBX_RENDER_MAX_THREADS 256
#define TBX_RENDER_MIN_CTAS 4
#define TBX_NT ((int)blockDim.x)
#define TBX_NW ((int)(blockDim.x >> 5))
#define TBX_EPC 8
#define TBX_MAX_RECTS 96
#define TBX_MAX_BIG 64 /* queue of large / sprite primitives of a group painted by several warps */

static __device__ const uint32_t d_bank[TBX_BANK_WORDS] = TBX_BANK_INIT;
/* ceil(65536 / s) for the sprite scale factors s = 1..15 */
static __device__ const uint32_t d_inv16[16] = {0, 65536, 32768, 21846, 16384, 13108, 10923, 9363, 8192, 7282, 6554, 5958, 5462, 5042, 4682, 4370};

template <int GAME> struct Traits;
template <> struct Traits<TBX_BREAKOUT> {
  typedef BrkCfg Cfg; typedef BrkTable Table; typedef BrkRec Rec;
  static constexpr int W = TBX_BRK_W, H = TBX_BRK_H, NS = BRK_N_SLOTS, RW = TBX_WORDS(BrkRec), NG = BRK_N_GROUPS;
  static __device__ __forceinline__ void step(const TbxAcc &S, const Cfg &c, const Table *t, int in) { brk_step(S, c, t, in); }
  static __device__ __forceinline__ void new_game(const TbxAcc &S, const Cfg &c, const Table *) { brk_new_game(S, c); }
  static __device__ __forceinline__ TbxPrim prim(const uint32_t *R, const Cfg &c, const Table *t, int s, int base) { return brk_prim_delta(R, c, t, s, base); }
  static __device__ __forceinline__ int base_id(const uint32_t *R, const Cfg &c, const Table *t) { return brk_base_id(R, c, t); }
  static __device__ __forceinline__ void group(int g, const uint32_t *R, const Table *t, int base, int &b, int &e, int &mode) { brk_group(g, R, t, base, b, e, mode); }
  static __device__ __forceinline__ void trim(int, const uint32_t *, const Cfg &, int, int &, int &) {}
  static __device__ __forceinline__ int digit_index(int s) { return s >= BRK_SLOT_SCORE && s < BRK_SLOT_BRICKS ? s - BRK_SLOT_SCORE : -1; } /* HUD digit slots */
  /* cheap estimate of the number of entries that differ from the base frame: the runs of dead bricks */
  template <class LD> static __device__ __forceinline__ int dense_hint(LD ld, const Cfg &c, const Table *t) { /* ld(w) = word w of the env */
    const int tbl = (int32_t)ld(TBX_W(TbxHdr, tbl));
    const Table &T = t[tbl];
    if (!(tbl == c.default_tbl && T.delta_ok)) return 1 << 20; /* not on base frame 1: every brick is an entry */
    int n = 0; /* runs of consecutive dead bricks = entries after brk_prim_delta's vertical merging (column ends ignored) */
    uint32_t carry = 0;
    for (int k = 0; k < 5; k++) {
      const uint32_t dead = T.all_mask[k] & ~ld(TBX_W(BrkRec, alive) + k);
      n += __popc(dead & ~((dead << 1) | carry));
      carry = dead >> 31;
    }
    return n;
  }
};
template <> struct Traits<TBX_SPACE_INVADERS> {
  typedef SiCfg Cfg; typedef int Table; typedef SiRec Rec;
  static constexpr int W = TBX_SI_W, H = TBX_SI_H, NS = SI_N_SLOTS, RW = TBX_WORDS(SiRec), NG = SI_N_GROUPS;
  static __device__ __forceinline__ void step(const TbxAcc &S, const Cfg &c, const Table *, int in) { si_step(S, c, in); }
  static __device__ __forceinline__ void new_game(const TbxAcc &S, const Cfg &c, const Table *) { si_new_game(S, c); }
  static __device__ __forceinline__ TbxPrim prim(const uint32_t *R, const Cfg &, const Table *, int s, int) { return si_prim(R, s); }
  static __device__ __forceinline__ int base_id(const uint32_t *, const Cfg &, const Table *) { return 0; }
  static __device__ __forceinline__ void group(int g, const uint32_t *, const Table *, int, int &b, int &e, int &mode) { si_group(g, b, e, mode); }
  static __device__ __forceinline__ void trim(int, const uint32_t *, const Cfg &, int, int &, int &) {}
  static __device__ __forceinline__ int digit_index(int s) { return s >= SI_SLOT_SCORE && s < SI_SLOT_SHIELDS ? s - SI_SLOT_SCORE : -1; }
  template <class LD> static __device__ __forceinline__ int dense_hint(LD, const Cfg &, const Table *) { return 0; } /* ~50 sprites, always: painted once each */
};
template <> struct Traits<TBX_AMIDAR> {
  typedef AmiCfg Cfg; typedef AmiTable Table; typedef AmiRec Rec;
  static constexpr int W = TBX_AMI_W, H = TBX_AMI_H, NS = AMI_N_SLOTS, RW = TBX_WORDS(AmiRec), NG = AMI_N_GROUPS;
  static __device__ __forceinline__ void step(const TbxAcc &S, const Cfg &c, const Table *t, int in) { ami_step(S, c, t, in); }
  static __device__ __forceinline__ void new_game(const TbxAcc &S, const Cfg &c, const Table *t) { ami_new_game(S, c, t); }
  static __device__ __forceinline__ TbxPrim prim(const uint32_t *R, const Cfg &c, const Table *t, int s, int base) { return ami_prim_delta(R, c, t, s, base); }
  static __device__ __forceinline__ int base_id(const uint32_t *R, const Cfg &c, const Table *t) { return ami_base_id(R, c, t); }
  static __device__ __forceinline__ void group(int g, const uint32_t *, const Table *, int, int &b, int &e, int &mode) { ami_group(g, b, e, mode); }
  /* Warp-cooperative narrowing of a group's slot range (every lane of the warp must call it): of the 31 x 32 maze
   * tiles only the rows whose packed words differ from the config board can differ from base frame 1 -- lane r
   * compares row r, a ballot gives the first and last such row.  (A superset: equal looks may hide behind unequal
   * tags; ami_prim_delta still decides per tile.) */
  static __device__ __forceinline__ void trim(int g, const uint32_t *R, const Cfg &c, int base, int &b, int &e) {
    if (g != 0 || base != 1) return;
    const int lane = threadIdx.x & 31;
    bool diff = false;
    if (lane < TBX_AMI_BH)
      diff = ((R[AMI_W(tiles) + 2 * lane] ^ c.board[lane][0]) | (R[AMI_W(tiles) + 2 * lane + 1] ^ c.board[lane][1])) != 0;
    const unsigned m = __ballot_sync(0xffffffffu, diff);
    if (m == 0) { e = b; return; }
    b = AMI_SLOT_TILES + 32 * (__ffs(m) - 1);
    e = AMI_SLOT_TILES + 32 * (32 - __clz(m));
  }
  static __device__ __forceinline__ int digit_index(int s) { return s >= AMI_SLOT_SCORE && s < AMI_N_SLOTS ? s - AMI_SLOT_SCORE : -1; }
  /* warp-cooperative (every lane calls it): tiles whose packed tag differs from the config board + painted boxes */
  template <class LD> static __device__ __forceinline__ int dense_hint(LD ld, const Cfg &c, const Table *) {
    const int lane = threadIdx.x & 31;
    int n = 0;
    if (lane < TBX_AMI_BH) {
      const uint32_t d0 = ld(AMI_W(tiles) + 2 * lane) ^ c.board[lane][0], d1 = ld(AMI_W(tiles) + 2 * lane + 1) ^ c.board[lane][1];
      n = __popc((d0 | (d0 >> 1)) & 0x55555555u) + __popc((d1 | (d1 >> 1)) & 0x55555555u);
    }
    return __reduce_add_sync(0xffffffffu, n) + __popc(ld(AMI_W(box_painted)));
  }
};

struct RenderArgs {
  const uint32_t *planes;
  int n, n_pad;
  const void *cfg, *tables;
  uint8_t *dst;
  size_t frame_bytes;
  const uint8_t *base[2];     /* base frames 0/1 in the canvas format: gray bytes, packed RGB or RGBA */
  const uint8_t *base_out[2]; /* INTER_AREA: their down-samples */
  const TbxAreaPlan *plan;    /* INTER_AREA */
  int band_rows;              /* native layouts: frame rows per CTA (blockIdx.y selects the band) */
  int smem_canvas, smem_rects; /* byte offsets into dynamic shared memory */
  /* dual mode (tbx_wrap.cuh): observation = INTER_AREA(max(frame(planes), frame(planes2))), written into slot
   * `stack_slot` of a ring of `stack_k` frames per env; envs flagged in reset_flags get the frame in every slot */
  const uint32_t *planes2;
  const uint8_t *reset_flags;
  size_t env_stride; /* bytes between the observations of consecutive envs (frame_bytes * stack_k) */
  int stack_k, stack_slot, tile_bytes;
  int stack_mode; /* envs flagged in reset_flags: 0 = the frame goes into every slot (FrameStack.reset), 1 = the other slots are zeroed (VecFrameStack) */
  /* native layouts, broadcast + patch (tbx_render_native.cuh): envs with more than dense_threshold entries (by the
   * game's cheap estimate) are not patched but appended to dense_list; the canvas kernel then repaints exactly those
   * (env_list / env_count != NULL: CTA b renders envs env_list[8b .. 8b+7], b < ceil(*env_count / 8)) */
  int32_t *dense_list;
  int *dense_count;
  uint8_t *dense_flag; /* [n]: 1 = left to the canvas kernel (written by dense_classify_kernel) */
  int dense_threshold;
  const int32_t *env_list;
  const int *env_count;
  const TbxDigitPatch *patches[2]; /* INTER_AREA: pre-resolved HUD digit patches per base frame, [slot * 10 + digit]; NULL = off */
  int tile_stride, warp_bytes, list_cap; /* INTER_AREA tile kernel (tbx_render_area.cuh): scratch row pitch, shared memory per warp */
};

/* The canvas is a byte array with PIX bytes per pixel: 1 = gray, 3 = packed RGB, 4 = RGBA.  `val` is the colour
 * as RGBA (r | g<<8 | b<<16 | a<<24) for PIX 3 and 4, the gray byte for PIX 1. */
template <int PIX> __device__ __forceinline__ void put_pixel(uint8_t *canvas, size_t pix, uint32_t val) {
  if (PIX == 1) canvas[pix] = (uint8_t)val;
  else if (PIX == 4) reinterpret_cast<uint32_t *>(canvas)[pix] = val;
  else { uint8_t *p = canvas + 3 * pix; p[0] = (uint8_t)val; p[1] = (uint8_t)(val >> 8); p[2] = (uint8_t)(val >> 16); }
}

struct Clip { int x0, y0, x1, y1; };
template <int W> __device__ __forceinline__ bool clip_prim(const TbxPrim &p, int r0, int r1, Clip &c) {
  c.x0 = max((int)p.x, 0); c.x1 = min((int)p.x + (int)p.w, W);
  c.y0 = max((int)p.y, r0); c.y1 = min((int)p.y + (int)p.h, r1);
  return p.h > 0 && c.x0 < c.x1 && c.y0 < c.y1;
}

/* one thread fills a small solid rectangle: 32-bit stores over the aligned middle of each row (4 gray pixels per
 * word; 4 RGB pixels = 3 words whose byte pattern repeats every 12 bytes), single pixels at the ragged ends */
template <int PIX, int W>
__device__ __forceinline__ void paint_small(uint8_t *canvas, int r0, const Clip &c, uint32_t val) {
  if (PIX == 4) {
    for (int y = c.y0; y < c.y1; y++) {
      uint32_t *row = reinterpret_cast<uint32_t *>(canvas) + (size_t)(y - r0) * W;
      for (int x = c.x0; x < c.x1; x++) row[x] = val;
    }
    return;
  }
  const int xa = min((c.x0 + 3) & ~3, c.x1), xb = max(c.x1 & ~3, xa);
  const uint32_t w0 = PIX == 1 ? (val & 255u) * 0x01010101u : ((val & 0xffffffu) | (val << 24));
  const uint32_t w1 = ((val >> 8) & 0xffffu) | (val << 16), w2 = ((val >> 16) & 0xffu) | (val << 8);
  for (int y = c.y0; y < c.y1; y++) {
    uint8_t *row = canvas + (size_t)(y - r0) * W * PIX;
    for (int x = c.x0; x < xa; x++) put_pixel<PIX>(row, x, val);
    for (int x = xa; x < xb; x += 4) {
      uint32_t *q = reinterpret_cast<uint32_t *>(row + x * PIX);
      q[0] = w0;
      if (PIX == 3) { q[1] = w1; q[2] = w2; }
    }
    for (int x = xb; x < c.x1; x++) put_pixel<PIX>(row, x, val);
  }
}

/* a whole warp paints one primitive (solid or sprite-masked), lanes over its clipped pixels */
template <int PIX, int W>
__device__ __forceinline__ void paint_coop(uint8_t *canvas, int r0, const Clip &c, int qx, int qy, uint32_t val, uint32_t q3,
                                           const uint32_t *rec, int lane) {
  /* lanes tile the rectangle as (32 >> lg) rows x (1 << lg) columns per pass: no divisions, no int<->float
   * conversions (those run on the quarter-rate XU pipe) */
  const int nw = c.x1 - c.x0, nh = c.y1 - c.y0;
  const int lg = nw > 16 ? 5 : nw > 8 ? 4 : nw > 4 ? 3 : nw > 2 ? 2 : nw > 1 ? 1 : 0;
  const int cpl = 1 << lg, rpp = 32 >> lg, sub = lane >> lg, cx = lane & (cpl - 1);
  const int bw = (q3 >> 16) & 255;
  if (bw == 0) {
    for (int xb = cx; xb < nw; xb += cpl)
      for (int yy = sub; yy < nh; yy += rpp) put_pixel<PIX>(canvas, (size_t)(c.y0 + yy - r0) * W + c.x0 + xb, val);
  } else {
    const uint32_t off = q3 & 0xffffu;
    const uint32_t *rows = (off & TBX_PRIM_STATE) ? rec + (off & 0x7fffu) : d_bank + off;
    const int sx = (q3 >> 24) & 15, sy = q3 >> 28;
    const uint32_t ix = d_inv16[sx], iy = d_inv16[sy]; /* v / s == (v * ceil(65536 / s)) >> 16 for v < 4096 */
    for (int xb = cx; xb < nw; xb += cpl) {
      const int px = c.x0 + xb - qx;
      const int sx_i = sx == 1 ? px : (int)(((uint32_t)px * ix) >> 16);
      for (int yy = sub; yy < nh; yy += rpp) {
        const int py = c.y0 + yy - qy;
        const int sy_i = sy == 1 ? py : (int)(((uint32_t)py * iy) >> 16);
        if ((rows[sy_i] >> (bw - 1 - sx_i)) & 1u) put_pixel<PIX>(canvas, (size_t)(c.y0 + yy - r0) * W + c.x0 + xb, val);
      }
    }
  }
}

/* dirty-rectangle list: rects[0..min(*n, TBX_MAX_RECTS)); *n > TBX_MAX_RECTS means "overflowed: everything is dirty" */
__device__ __forceinline__ void push_rect(int4 *rects, int *n, int4 r) {
  int slot = atomicAdd(n, 1);
  if (slot < TBX_MAX_RECTS) rects[slot] = r;
}

/* Paint every draw-list group of one env that differs from base frame `base` into canvas rows [r0,r1), in draw
 * order, and append the painted areas to the dirty list: one bounding box per warp pass of a parallel group (32
 * consecutive slots are spatially close: brick columns, a tile row), one rectangle per primitive of the in-order
 * group.  All threads of the CTA must call this; it ends with a barrier. */
template <int GAME, int PIX>
__device__ __forceinline__ void paint_env(const uint32_t *R, const typename Traits<GAME>::Cfg &cfg, const typename Traits<GAME>::Table *tables,
                                          int base, uint8_t *canvas, int r0, int r1, int4 *rects, int *n_rects, uint4 *bigs, int *n_big) {
  typedef Traits<GAME> T;
  constexpr int W = T::W;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  /* Barriers: painting order between two consecutive groups must be enforced across warps unless both run on
   * warp 0 only (an in-order group, or a parallel group of at most 32 slots) -- then program order does it --
   * or the earlier group is flagged disjoint from the next (TBX_GROUP_NOSYNC). */
  bool have_prev = false, prev_multi = false, prev_nosync = false;
  for (int g = 0; g < T::NG; g++) {
    int gb, ge, gmode;
    T::group(g, R, tables, base, gb, ge, gmode);
    T::trim(g, R, cfg, base, gb, ge);
    if (gb >= ge) { prev_nosync = false; continue; } /* empty group (uniform across the CTA); its neighbour's flag does not carry over */
    const bool cur_multi = !(gmode & TBX_GROUP_SERIAL) && (ge - gb) > 32;
    if (have_prev && (prev_multi || cur_multi) && !prev_nosync) __syncthreads();
    else if (have_prev) __syncwarp(); /* warp 0 after warp 0: orders the other lanes' stores of the earlier group before this one's */
    have_prev = true;
    prev_multi = cur_multi;
    prev_nosync = (gmode & TBX_GROUP_NOSYNC) != 0 && !cur_multi; /* a multi-warp group resets its queue: always fenced */
    if (!(gmode & TBX_GROUP_SERIAL)) {
      for (int s0 = gb; s0 < ge; s0 += TBX_NT) {
        const int s = s0 + tid;
        TbxPrim p = tbx_prim_none();
        if (s < ge) p = T::prim(R, cfg, tables, s, base);
        Clip c;
        const bool ok = clip_prim<W>(p, r0, r1, c);
        if (!__any_sync(0xffffffffu, ok)) continue;
        const uint32_t val = PIX == 1 ? tbx_luma(p.color) : p.color;
        const bool small = ok && p.bw == 0 && (c.x1 - c.x0) * (c.y1 - c.y0) <= 512; /* up to a column of merged dead bricks: one thread, word stores */
        if (small) paint_small<PIX, W>(canvas, r0, c, val);
        __syncwarp(); /* lane-painted rectangles before the warp-painted ones of the same pass */
        const uint32_t w0 = (uint16_t)p.x | ((uint32_t)(uint16_t)p.y << 16), w1 = (uint16_t)p.w | ((uint32_t)(uint16_t)p.h << 16);
        const uint32_t w3 = (uint32_t)p.off | ((uint32_t)p.bw << 16) | ((uint32_t)p.scale << 24);
        bool deferred = false;
        if (cur_multi && ok && !small) { /* a group spread over several warps: queue it, every warp takes its share below */
          const int k = atomicAdd(n_big, 1);
          if (k < TBX_MAX_BIG) { bigs[k] = make_uint4(w0, w1, val, w3); deferred = true; }
        }
        unsigned big = __ballot_sync(0xffffffffu, ok && !small && !deferred);
        if (big) {
          while (big) {
            const int l = __ffs(big) - 1;
            big &= big - 1;
            TbxPrim q;
            const uint32_t q0 = __shfl_sync(0xffffffffu, w0, l), q1 = __shfl_sync(0xffffffffu, w1, l);
            const uint32_t qv = __shfl_sync(0xffffffffu, val, l), q3 = __shfl_sync(0xffffffffu, w3, l);
            q.x = (int16_t)(q0 & 0xffffu); q.y = (int16_t)(q0 >> 16); q.w = (int16_t)(q1 & 0xffffu); q.h = (int16_t)(q1 >> 16);
            Clip qc;
            clip_prim<W>(q, r0, r1, qc);
            paint_coop<PIX, W>(canvas, r0, qc, q.x, q.y, qv, q3, R, lane);
          }
        }
        /* dirty area of this warp pass (hardware integer warp reductions): its bounding box when the primitives
         * fill it densely (bricks, tiles), else one rectangle per primitive (sprites spread over a formation) */
        const int bx0 = __reduce_min_sync(0xffffffffu, ok ? c.x0 : 32767), by0 = __reduce_min_sync(0xffffffffu, ok ? c.y0 : 32767);
        const int bx1 = __reduce_max_sync(0xffffffffu, ok ? c.x1 : -1), by1 = __reduce_max_sync(0xffffffffu, ok ? c.y1 : -1);
        const int covered = __reduce_add_sync(0xffffffffu, ok ? (c.x1 - c.x0) * (c.y1 - c.y0) : 0);
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        const int room = __shfl_sync(0xffffffffu, TBX_MAX_RECTS - 40 - *(volatile int *)n_rects, 0); /* keep room for the later groups */
        if ((bx1 - bx0) * (by1 - by0) <= 2 * covered || __popc(m) > room) {
          if (lane == 0) push_rect(rects, n_rects, make_int4(bx0, by0, bx1, by1));
        } else {
          int slot0 = 0;
          if (lane == 0) slot0 = atomicAdd(n_rects, __popc(m));
          slot0 = __shfl_sync(0xffffffffu, slot0, 0);
          const int slot = slot0 + __popc(m & ((1u << lane) - 1u));
          if (ok && slot < TBX_MAX_RECTS) rects[slot] = make_int4(c.x0, c.y0, c.x1, c.y1);
        }
      }
      if (cur_multi) { /* the queued large / sprite primitives of this conflict-free group, one warp each, round robin */
        __syncthreads();
        const int nb = min(*n_big, TBX_MAX_BIG);
        __syncthreads();
        if (tid == 0) *n_big = 0; /* the next queueing group starts behind a barrier */
        for (int i = wid; i < nb; i += TBX_NW) {
          const uint4 q4 = bigs[i];
          TbxPrim q;
          q.x = (int16_t)(q4.x & 0xffffu); q.y = (int16_t)(q4.x >> 16); q.w = (int16_t)(q4.y & 0xffffu); q.h = (int16_t)(q4.y >> 16);
          Clip qc;
          clip_prim<W>(q, r0, r1, qc);
          paint_coop<PIX, W>(canvas, r0, qc, q.x, q.y, q4.z, q4.w, R, lane);
        }
      }
    } else if (wid == 0) {
      /* in order: lane l builds primitive gb + 32*batch + l, then the warp paints them one at a time */
      for (int s0 = gb; s0 < ge; s0 += 32) {
        const int s = s0 + lane;
        TbxPrim p = tbx_prim_none();
        if (s < ge) p = T::prim(R, cfg, tables, s, base);
        Clip c;
        const bool ok = clip_prim<W>(p, r0, r1, c);
        const uint32_t val = PIX == 1 ? tbx_luma(p.color) : p.color;
        unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m == 0) continue;
        int slot0 = 0;
        if (lane == 0) slot0 = atomicAdd(n_rects, __popc(m));
        slot0 = __shfl_sync(0xffffffffu, slot0, 0);
        const int slot = slot0 + __popc(m & ((1u << lane) - 1u));
        if (ok && slot < TBX_MAX_RECTS) rects[slot] = make_int4(c.x0, c.y0, c.x1, c.y1);
        const uint32_t w0 = (uint16_t)p.x | ((uint32_t)(uint16_t)p.y << 16), w1 = (uint16_t)p.w | ((uint32_t)(uint16_t)p.h << 16);
        const uint32_t w3 = (uint32_t)p.off | ((uint32_t)p.bw << 16) | ((uint32_t)p.scale << 24);
        while (m) {
          const int l = __ffs(m) - 1;
          m &= m - 1;
          TbxPrim q;
          const uint32_t q0 = __shfl_sync(0xffffffffu, w0, l), q1 = __shfl_sync(0xffffffffu, w1, l);
          const uint32_t qv = __shfl_sync(0xffffffffu, val, l), q3 = __shfl_sync(0xffffffffu, w3, l);
          q.x = (int16_t)(q0 & 0xffffu); q.y = (int16_t)(q0 >> 16); q.w = (int16_t)(q1 & 0xffffu); q.h = (int16_t)(q1 >> 16);
          Clip qc;
          clip_prim<W>(q, r0, r1, qc);
          paint_coop<PIX, W>(canvas, r0, qc, q.x, q.y, qv, q3, R, lane);
          __syncwarp();
        }
      }
    }
  }
  __syncthreads();
}

/* copy rows [r0,r1) of a base frame into the canvas (full initialisation) */
template <int PIX, int W>
__device__ __forceinline__ void load_canvas(uint8_t *canvas, const uint8_t *base, int r0, int r1) {
  const uint4 *src = reinterpret_cast<const uint4 *>(base + (size_t)r0 * W * PIX);
  uint4 *dst = reinterpret_cast<uint4 *>(canvas);
  const int n16 = (r1 - r0) * W * PIX / 16;
#pragma unroll 4
  for (int i = threadIdx.x; i < n16; i += TBX_NT) dst[i] = __ldg(src + i);
}
/* undo one env's painting: re-copy the dirty rectangles (whole 16-byte chunks) from the base frame */
template <int PIX, int W>
__device__ __forceinline__ void restore_canvas(uint8_t *canvas, const uint8_t *base, int r0, int r1, const int4 *rects, int n) {
  if (n > TBX_MAX_RECTS) { load_canvas<PIX, W>(canvas, base, r0, r1); return; }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int i = wid; i < n; i += TBX_NW) {
    const int4 rc = rects[i];
    if (rc.z <= rc.x) continue;
    const int b0 = (rc.x * PIX) & ~15, b1 = (rc.z * PIX + 15) & ~15, nch = (b1 - b0) >> 4;
    const int nh = rc.w - rc.y;
    const int lg = nch > 16 ? 5 : nch > 8 ? 4 : nch > 4 ? 3 : nch > 2 ? 2 : nch > 1 ? 1 : 0;
    const int cpl = 1 << lg, rpp = 32 >> lg, sub = lane >> lg, cx = lane & (cpl - 1);
    for (int ch = cx; ch < nch; ch += cpl)
      for (int yy = sub; yy < nh; yy += rpp) {
        const size_t off = (size_t)(rc.y + yy) * W * PIX + b0 + 16 * ch;
        *reinterpret_cast<uint4 *>(canvas + off - (size_t)r0 * W * PIX) = __ldg(reinterpret_cast<const uint4 *>(base + off));
      }
  }
}

/* MODE: TBX_OBS_RGBA (0), TBX_OBS_RGB (1), TBX_OBS_GRAY (2) */
template <int GAME, int MODE>
__global__ void __launch_bounds__(TBX_RENDER_MAX_THREADS, TBX_RENDER_MIN_CTAS) render_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ typename Traits<GAME>::Cfg cfg_c) {
  /* The pool's config travels as a kernel parameter: warp-uniform reads of it (colours) come from the constant bank
   * instead of global memory. */
  typedef Traits<GAME> T;
  constexpr int W = T::W, H = T::H, RW = T::RW;
  constexpr int PIX = MODE == 0 ? 4 : MODE == 1 ? 3 : 1; /* canvas bytes per pixel = output bytes per pixel */
  extern __shared__ uint4 smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>(smem_raw);
  uint32_t *recs = reinterpret_cast<uint32_t *>(smem);
  uint8_t *canvas = smem + a.smem_canvas;
  int4 *rect_buf = reinterpret_cast<int4 *>(smem + a.smem_rects); /* two lists, used alternately */
  int *rect_n = reinterpret_cast<int *>(rect_buf + 2 * TBX_MAX_RECTS);
  int *env_base = rect_n + 2; /* base frame id of each env of the chunk */
  int *n_big = env_base + 2 * TBX_EPC;
  uint4 *big_buf = reinterpret_cast<uint4 *>(rect_n + 32);
  const typename T::Cfg &cfg = cfg_c;
  const typename T::Table *tables = (const typename T::Table *)a.tables;
  const int tid = threadIdx.x;
  const int e0 = blockIdx.x * TBX_EPC;
  const int ne = min(TBX_EPC, (a.env_count ? *a.env_count : a.n) - e0);
  if (ne <= 0) return; /* env-list mode: nothing (left) to repaint */
  int *env_id = env_base + TBX_EPC; /* the env each slot of the chunk renders */
  if (tid < TBX_EPC) env_id[tid] = a.env_list ? (tid < ne ? a.env_list[e0 + tid] : 0) : e0 + tid;
  __syncthreads();

  /* coalesced load of the chunk's state words: thread -> (word, env) with env fastest */
  for (int i = tid; i < RW * TBX_EPC; i += TBX_NT) {
    int w = i / TBX_EPC, j = i - w * TBX_EPC;
    if (j < ne) recs[j * RW + w] = a.planes[(size_t)w * a.n_pad + env_id[j]];
  }
  if (tid < 2) rect_n[tid] = 0;
  if (tid == 2) *n_big = 0;
  __syncthreads();

  if (tid < ne) env_base[tid] = T::base_id(recs + tid * RW, cfg, tables);
  __syncthreads();

  /* The canvas holds the output format, so the painted band IS the output band and leaves through the TMA engine --
   * one bulk shared -> global copy per env (cp.async.bulk), no per-thread load/store instructions. */
  const int r0 = blockIdx.y * a.band_rows, r1 = min(H, r0 + a.band_rows);
  int canvas_base = -1;
#pragma unroll 1 /* the body is large: unrolled over the 8 envs it no longer fits the instruction cache (measured: 2x slower) */
  for (int j = 0; j < ne; j++) {
    const uint32_t *R = recs + j * RW;
    const int base = env_base[j];
    int4 *rects = rect_buf + (j & 1) * TBX_MAX_RECTS;
    int *n_rects = rect_n + (j & 1);
    uint8_t *out = a.dst + (size_t)env_id[j] * a.frame_bytes;
    if (canvas_base != base) load_canvas<PIX, W>(canvas, (base ? a.base[1] : a.base[0]), r0, r1);
    else restore_canvas<PIX, W>(canvas, (base ? a.base[1] : a.base[0]), r0, r1, rect_buf + ((j - 1) & 1) * TBX_MAX_RECTS, rect_n[(j - 1) & 1]);
    canvas_base = base;
    __syncthreads();
    if (tid == 0) rect_n[(j - 1) & 1] = 0;
    paint_env<GAME, PIX>(R, cfg, tables, base, canvas, r0, r1, rects, n_rects, big_buf, n_big);
    /* every thread makes its canvas writes visible to the async proxy; the canvas may be touched again once the
     * engine has read it.  (Half of all stall samples of the sprite-heavy games sit in this wait; two half-height
     * canvases painted alternately were measured and are slower -- the per-band fixed work doubles.) */
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(canvas);
      const uint32_t nbytes = (uint32_t)((r1 - r0) * W * PIX);
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out + (size_t)r0 * W * PIX), "r"(saddr), "r"(nbytes) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    __syncthreads(); /* the canvas is restored next */
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); /* all bands have left */
}

} /* namespace tbxk */
#endif
