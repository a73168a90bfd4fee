/* tbx_direct.h -- DIRECT evaluation of the INTER_AREA (WarpFrame, 84x84 gray) observation: closed forms per game
 * instead of "paint a canvas, then resolve it".
 *
 * The reference produces the observation as get_state() (toybox/envs/atari/base.py:109) followed by
 * cv2.resize(..., INTER_AREA) (baselines/baselines/common/atari_wrappers.py:243).  An output pixel is
 *     round( sum_k yalpha[k][dy] * ( sum_t xalpha[t][dx] * src[ys0[dy] + k][xs0[dx] + t] ) )      (f32, this order)
 * and the native frame `src` is never needed as a whole:
 *   - where the frame is a regular GRID of cells whose rows repeat (Breakout's brick wall), the inner sum of one
 *     source row depends on the alive bits of at most two neighbouring cells: it is a table look-up (host-built with
 *     the very same f32 operations), and one look-up serves every source row of the cell row;
 *   - where a few small MOVERS (paddle, balls) sit on top, only the output pixels their rectangles feed are evaluated,
 *     tap by tap, with an analytic painter's algorithm: base pixel, then grid cell, then the movers in draw order;
 *   - HUD digits are pre-resolved patches (TbxDigitPatch), everything else is the pre-computed down-sample of the base
 *     frame.
 * The functions here are TBX_HD: the kernels of tbx_render_direct.cuh and the CPU-tier emulation (tests/emu) run the
 * same code.  Envs the closed forms do not cover (custom brick tables, movers inside the HUD rows) are rendered by the
 * general tile kernel (tbx_render_area.cuh).
 */
#ifndef TBX_DIRECT_H
#define TBX_DIRECT_H
#include "tbx_breakout.h"
#include "tbx_space_invaders.h"
#include "tbx_amidar.h"

/* a clipped rectangle of the draw list with its gray value; x0 >= x1: empty */
struct TbxMover { int x0, y0, x1, y1; uint32_t gray; };

/* ------------------------------------------------------------------ Breakout */
#define TBX_BD_MAX_STATIC 16
#define TBX_BD_MAX_CLS 8
#define BRK_N_MOVERS (1 + TBX_BRK_MAX_BALLS) /* paddle, balls in draw order */
typedef struct TbxBrkDirect {
  int32_t ok;                    /* 0: this (config, output size) pair is rendered by the tile kernel */
  int32_t ncols, nrows;          /* the default table is a grid of ncols x nrows bricks, index = col * nrows + row */
  int32_t wx0, wy0, bw, bh;      /* origin of the grid and brick size in pixels */
  int32_t wdy0, wdy1;            /* output rows fed by the wall's source rows (inclusive) */
  int32_t hud_dyhi;              /* last output row fed by a HUD digit row */
  int32_t n_static, _pad;
  uint32_t paddle_gray, ball_gray;
  uint8_t xcol[TBX_AREA_MAX_SRC]; /* brick column of source column x, 255 = none */
  uint8_t yrow[TBX_AREA_MAX_SRC]; /* brick row of source row y, 255 = none */
  uint8_t col0[TBX_AREA_MAX_DST]; /* per output column: the taps touch brick columns col0 and col0 + 1 only */
  uint8_t dyrows[TBX_AREA_MAX_DST]; /* per output row: mask of the brick rows its taps touch */
  uint8_t hsel[TBX_AREA_MAX_DST][TBX_AREA_MAX_TAPS]; /* per output row and tap: H row -- < nrows: brick row, else static row (- nrows) */
  uint32_t wordcols[32];          /* per output word (4 columns): mask of the brick columns that feed it */
  uint8_t brickgray[TBX_BRK_MAX_BRICKS];
  uint32_t inv32[TBX_AREA_MAX_DST + 1]; /* ceil(2^32 / n) for n >= 2: i / n == umulhi(i, inv32[n]) for the small i used here */
  alignas(16) float hlut[TBX_BRK_MAX_ROWS][4][TBX_AREA_MAX_DST];  /* [brick row][alive(col0) | alive(col0 + 1) << 1][dx] */
  alignas(16) float hstatic[TBX_BD_MAX_STATIC][TBX_AREA_MAX_DST]; /* horizontal sums of the base-frame-0 rows around the wall */
  /* base frame 0 by row classes: its rows fall into a few classes of identical rows (background, borders, HUD band), so the
   * movers' source windows read a 2 KB table in shared memory instead of the 38 KB frame.  n_cls == 0: more classes than fit */
  int32_t n_cls, _pad2[3];
  uint8_t rowcls[TBX_BRK_H];
  alignas(16) uint8_t clsrows[TBX_BD_MAX_CLS * TBX_BRK_W + 16];
} TbxBrkDirect;

/* THE SHARED-MEMORY IMAGE of the Breakout direct kernel: every table its per-env code reads, laid out on the host exactly as the
 * kernel wants it (tbx::build_brk_img, one per (config, output size)) and copied whole, by one bulk copy, at the start of its shared
 * memory.  The fixed-size tables come first, at offsets that depend on TY only (constants in the kernel), then the tables sized by
 * the output size and the config (brk_img_layout).  Every offset is a multiple of 16. */
#define TBX_A16(v) (((v) + 15) & ~15)
#define TBX_BRK_DIG_SLOTS 6  /* digit slots whose patches are kept in the image: score digits 0..3, lives digits 0..1 */
#define TBX_BRK_DIG_WORDS 13 /* header word + up to 48 pixels: the first 52 bytes of the TbxDigitPatch */
#define TBX_BRK_DIG_BYTES (TBX_BRK_DIG_SLOTS * 10 * TBX_BRK_DIG_WORDS * 4)
#define TBX_BI_FLAGS 0                                                          /* int32: 1 = every cached slot's patches fit 48 pixels */
#define TBX_BI_DIG 16                                                           /* uint32 [6 slots x 10 digits][13] */
#define TBX_BI_ROWCLS (TBX_BI_DIG + TBX_A16(TBX_BRK_DIG_BYTES))                 /* TbxBrkDirect.rowcls */
#define TBX_BI_INV (TBX_BI_ROWCLS + TBX_A16(TBX_BRK_H))                         /* .inv32 */
#define TBX_BI_XDLO (TBX_BI_INV + TBX_A16(4 * (TBX_AREA_MAX_DST + 1)))          /* plan xdlo / xdhi / ydlo / ydhi over the frame's W or H */
#define TBX_BI_XDHI (TBX_BI_XDLO + TBX_A16(TBX_BRK_W))
#define TBX_BI_YDLO (TBX_BI_XDHI + TBX_A16(TBX_BRK_W))
#define TBX_BI_YDHI (TBX_BI_YDLO + TBX_A16(TBX_BRK_H))
#define TBX_BI_XCOL (TBX_BI_YDHI + TBX_A16(TBX_BRK_H))                          /* .xcol over W */
#define TBX_BI_YROW (TBX_BI_XCOL + TBX_A16(TBX_BRK_W))                          /* .yrow over H */
#define TBX_BI_BGRAY (TBX_BI_YROW + TBX_A16(TBX_BRK_H))                         /* .brickgray */
#define TBX_BI_WORDCOLS (TBX_BI_BGRAY + TBX_A16(TBX_BRK_MAX_BRICKS))            /* .wordcols */
#define TBX_BI_COL0 (TBX_BI_WORDCOLS + 4 * 32)                                  /* .col0 */
#define TBX_BI_DYROWS (TBX_BI_COL0 + TBX_A16(TBX_AREA_MAX_DST))                 /* .dyrows */
#define TBX_BI_HSEL (TBX_BI_DYROWS + TBX_A16(TBX_AREA_MAX_DST))                 /* .hsel as [MAX_DST][TY] */
#define TBX_BI_FIXED(ty) (TBX_BI_HSEL + TBX_A16(TBX_AREA_MAX_DST * (ty)))
/* pitch of the plan's per-pixel tables in the image */
TBX_HD int brk_plan_pitch(int dw, int dh) { return ((dw > dh ? dw : dh) + 3) & ~3; }
struct TbxBrkImgLayout {
  int base1;   /* uint8 [dh][dw]: the down-sample of base frame 1 (every brick alive) */
  int plan;    /* float xalpha [TX][ps], yalpha [TY][ps]; uint16 xs0 [ps], ys0 [ps] (ps = brk_plan_pitch, clamped to dw - 1 / dh - 1) */
  int hlut;    /* float [nrows x 4][hs]: .hlut */
  int hstatic; /* float [n_static][hs]: the rows of .hstatic in use */
  int cls;     /* uint8 [n_cls][W] + 16 bytes of slack: the classes of .clsrows in use */
  int bytes;
};
TBX_HD TbxBrkImgLayout brk_img_layout(int tx, int ty, int dw, int dh, int nrows, int n_static, int n_cls) {
  const int ps = brk_plan_pitch(dw, dh), hs = (dw + 3) & ~3;
  TbxBrkImgLayout L;
  L.base1 = TBX_BI_FIXED(ty);
  L.plan = L.base1 + TBX_A16(dw * dh);
  L.hlut = L.plan + TBX_A16((tx + ty) * ps * 4 + 2 * ps * 2);
  L.hstatic = L.hlut + TBX_A16(nrows * 4 * hs * 4);
  L.cls = L.hstatic + TBX_A16(n_static * hs * 4);
  L.bytes = L.cls + TBX_A16(n_cls * TBX_BRK_W + 16);
  return L;
}

/* paddle (m == 0) or ball m - 1 as a clipped rectangle */
TBX_HD TbxMover brk_mover(const uint32_t *R, const BrkCfg &c, uint32_t paddle_gray, uint32_t ball_gray, int m) {
  TbxMover v; v.x0 = v.y0 = v.x1 = v.y1 = 0; v.gray = m == 0 ? paddle_gray : ball_gray;
  if (m < 0 || m >= BRK_N_MOVERS) return v;
  const TbxPrim p = brk_prim(R, c, (const BrkTable *)0, m == 0 ? BRK_SLOT_PADDLE : BRK_SLOT_BALLS + m - 1); /* these slots never read the tables */
  if (p.h <= 0) return v;
  const int x0 = p.x < 0 ? 0 : p.x, y0 = p.y < 0 ? 0 : p.y;
  const int x1 = p.x + p.w > TBX_BRK_W ? TBX_BRK_W : p.x + p.w, y1 = p.y + p.h > TBX_BRK_H ? TBX_BRK_H : p.y + p.h;
  if (x0 >= x1 || y0 >= y1) return v;
  v.x0 = x0; v.y0 = y0; v.x1 = x1; v.y1 = y1;
  return v;
}

/* tbx_d2i's contract (truncate, saturate to +-2^29, NaN -> 0) as one saturating conversion and two integer clamps: on the
 * device cvt.rzi.s32.f64 already saturates to the int32 range and maps NaN to 0; the host restates that conversion */
TBX_HD int tbx_d2i_sat(double v) {
#if defined(__CUDA_ARCH__)
  const int i = __double2int_rz(v);
  return min(max(i, -536870912), 536870912);
#else
  const int i = !(v == v) ? 0 : v >= 2147483647.0 ? 2147483647 : v <= -2147483648.0 ? (-2147483647 - 1) : (int)v;
  return i < -536870912 ? -536870912 : i > 536870912 ? 536870912 : i;
#endif
}

/* brk_mover read straight from the record (any word stride), without the draw-list primitive: the same rectangle for every
 * input.  tbx_prim_rect clips to +-30000 and keeps the extent in 16 bits, so an extent above 32767 after that clip wraps
 * negative and the mover draws nothing; the rest of its clipping is the canvas clip below. */
TBX_HD TbxMover brk_mover_rec(const TbxAcc &S, uint32_t paddle_gray, uint32_t ball_gray, int m) {
  TbxMover v; v.x0 = v.y0 = v.x1 = v.y1 = 0; v.gray = m == 0 ? paddle_gray : ball_gray;
  if (m < 0 || m >= BRK_N_MOVERS || (m > 0 && m > S.ldi(BRK_W(n_balls)))) return v;
  int x, y, w, h;
  if (m == 0) {
    const double pw = S.ldd(BRK_W(paddle_width));
    x = tbx_d2i_sat(tbx_dsub(S.ldd(BRK_W(paddle_px)), tbx_dmul(pw, 0.5)));
    y = tbx_d2i_sat(tbx_dsub(S.ldd(BRK_W(paddle_py)), BRK_PADDLE_HALF_H));
    w = tbx_d2i_sat(pw); h = 3;
  } else {
    const double r = S.ldd(BRK_W(ball_radius));
    const int b = BRK_W(ball) + 8 * (m - 1);
    x = tbx_d2i_sat(tbx_dsub(S.ldd(b), r));
    y = tbx_d2i_sat(tbx_dsub(S.ldd(b + 2), r));
    w = h = tbx_d2i_sat(tbx_dmul(r, 2.0));
  }
  /* |x|, |w| <= 2^29: x + w does not overflow; w <= 0 leaves x1 <= x0 */
  const int x0 = x < 0 ? 0 : x, y0 = y < 0 ? 0 : y;
  const int x1 = x + w > TBX_BRK_W ? TBX_BRK_W : x + w, y1 = y + h > TBX_BRK_H ? TBX_BRK_H : y + h;
  const int ex = (x + w > 30000 ? 30000 : x + w) - (x < -30000 ? -30000 : x), ey = (y + h > 30000 ? 30000 : y + h) - (y < -30000 ? -30000 : y);
  if (x0 >= x1 || y0 >= y1 || ex > 32767 || ey > 32767) return v;
  v.x0 = x0; v.y0 = y0; v.x1 = x1; v.y1 = y1;
  return v;
}

/* alive bits of brick column c (bit r = row r) */
TBX_HD uint32_t brk_col_bits(const uint32_t *alive, int nrows, int c) {
  const int i0 = c * nrows, w = i0 >> 5, s = i0 & 31;
  const uint32_t lo = alive[w], hi = w < 4 ? alive[w + 1] : 0u;
  const uint32_t v = s ? (lo >> s) | (hi << (32 - s)) : lo;
  return v & ((1u << nrows) - 1u);
}
/* ... the same from a record of any word stride, the alive words starting at word w0 */
TBX_HD uint32_t brk_col_bits(const TbxAcc &S, int w0, int nrows, int c) {
  const int i0 = c * nrows, w = i0 >> 5, s = i0 & 31;
  const uint32_t lo = S.ld(w0 + w), hi = w < 4 ? S.ld(w0 + w + 1) : 0u;
  const uint32_t v = s ? (lo >> s) | (hi << (32 - s)) : lo;
  return v & ((1u << nrows) - 1u);
}

/* gray value of native-frame pixel (x, y): base frame 0, then the brick grid, then the movers in `near` in draw order */
TBX_HD uint32_t brk_direct_src(const TbxBrkDirect &A, const uint8_t *base0, const uint32_t *alive, const TbxMover *mv, uint32_t near, bool wall,
                               int x, int y) {
  uint32_t v = base0[y * TBX_BRK_W + x];
  if (wall) {
    const uint32_t c = A.xcol[x], r = A.yrow[y];
    if ((c | r) != 255u) { /* both are < 255: a brick cell */
      const uint32_t i = c * (uint32_t)A.nrows + r;
      if ((alive[i >> 5] >> (i & 31)) & 1u) v = A.brickgray[i];
    }
  }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int m = 0; m < BRK_N_MOVERS; m++)
    if ((near >> m) & 1u)
      if ((unsigned)(x - mv[m].x0) < (unsigned)(mv[m].x1 - mv[m].x0) && (unsigned)(y - mv[m].y0) < (unsigned)(mv[m].y1 - mv[m].y0)) v = mv[m].gray;
  return v;
}

/* one output pixel, every tap evaluated analytically (zero-padded TX x TY taps in cv2's order) */
template <int TX, int TY>
TBX_HD uint8_t brk_direct_pixel(const TbxBrkDirect &A, const TbxAreaPlan &pl, const uint8_t *base0, const uint32_t *alive, const TbxMover *mv, uint32_t near,
                                bool wall, int dx, int dy) {
  const int xs = pl.xs0[dx], ys = pl.ys0[dy];
  float acc = 0.0f;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int k = 0; k < TY; k++) {
    const int y = ys + k < TBX_BRK_H ? ys + k : TBX_BRK_H - 1; /* surplus taps carry zero weights: any in-frame pixel will do */
    float h = 0.0f;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < TX; t++) {
      const int x = xs + t < TBX_BRK_W ? xs + t : TBX_BRK_W - 1;
      const float p = tbx_fmul(tbx_u8f(brk_direct_src(A, base0, alive, mv, near, wall, x, y)), pl.xalpha[t][dx]);
      h = t == 0 ? p : tbx_fadd(h, p);
    }
    const float bh = tbx_fmul(pl.yalpha[k][dy], h);
    acc = k == 0 ? bh : tbx_fadd(acc, bh);
  }
  const int iv = tbx_f2i_rn_small(acc);
  return (uint8_t)(iv < 0 ? 0 : iv > 255 ? 255 : iv);
}

/* the wall: horizontal sum of brick row r at output column dx from the row's alive mask (bit c = column c alive) */
TBX_HD float brk_direct_h(const TbxBrkDirect &A, int r, uint32_t rowmask, int dx) { return A.hlut[r][(rowmask >> A.col0[dx]) & 3u][dx]; }
/* ... and the output pixel from the H rows: hdyn[r * hstride + dx] holds brk_direct_h of brick row r */
template <int TY>
TBX_HD uint8_t brk_direct_wall_pixel(const TbxBrkDirect &A, const TbxAreaPlan &pl, const float *hdyn, int hstride, int dx, int dy) {
  float acc = 0.0f;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int k = 0; k < TY; k++) {
    const int sel = A.hsel[dy][k];
    const float h = sel < A.nrows ? hdyn[sel * hstride + dx] : A.hstatic[sel - A.nrows][dx];
    const float bh = tbx_fmul(pl.yalpha[k][dy], h);
    acc = k == 0 ? bh : tbx_fadd(acc, bh);
  }
  const int iv = tbx_f2i_rn_small(acc);
  return (uint8_t)(iv < 0 ? 0 : iv > 255 ? 255 : iv);
}

/* HUD digit k (0 = least significant) of a field value: -1 = not shown (tbx_prim_digit) */
TBX_HD int tbx_digit_at(int value, int k) {
  uint32_t q = value < 0 ? 0u : (uint32_t)value;
  for (int i = 0; i < k && q; i++) q /= 10u;
  if (k > 0 && q == 0) return -1;
  return (int)(q % 10u);
}

/* ------------------------------------------------------------------ sparse sprites on a plain base (Space Invaders)
 * The frame is the base frame (black + ground line) plus ~50 small entries of the draw list.  An entry whose output
 * footprint meets no other entry's ("simple") and lies on plain background is the only thing that differs from the base
 * there: if it is a 16-bit-wide bank sprite at scale 1 in one of its usual colours, its output pixels are a PRE-RESOLVED
 * PATCH that depends on the sprite and on (x mod px_period, y mod py_period) only -- INTER_AREA's tap pattern repeats
 * every px_period source columns / py_period source rows (84 x 84 from 320 x 210: 80 and 5).  Everything else (shields,
 * whose bits live in the state; lasers; entries that touch each other) is evaluated pixel by pixel: the TX x TY source
 * window is built as packed bytes from the base frame and the non-simple entries in draw order, then resolved in cv2's
 * tap order. */
#define TBX_SD_MAX_ENTRIES 72
#define TBX_SD_MAX_SETS 16
#define TBX_SC_MAX_COLS 32
#define TBX_SC_MAX_ROWS 4
#define TBX_SP_MAX_W 6
#define TBX_SP_MAX_H 5
typedef struct TbxSpritePatch { uint8_t w, h; uint8_t px[TBX_SP_MAX_W * TBX_SP_MAX_H]; } TbxSpritePatch; /* 32 bytes; pixel (r, c) at px[r * TBX_SP_MAX_W + c] */
typedef struct TbxSiDirect {
  int32_t ok;
  int32_t n_sets;                /* (sprite, gray) pairs with patch tables; 0: no patches (every entry is evaluated) */
  int32_t px_period, py_period;  /* source period of the tap pattern per axis */
  int32_t ox_period, oy_period;  /* output pixels per period */
  int32_t bg_gray, _pad;
  uint32_t inv_px, inv_py;       /* ceil(2^32 / period) (0 when the period is 1): v / period == umulhi(v, inv) for coordinates */
  uint16_t set_off[TBX_SD_MAX_SETS];  /* bank offset of the set's sprite */
  uint8_t set_gray[TBX_SD_MAX_SETS];
  uint8_t set_h[TBX_SD_MAX_SETS];     /* sprite rows (10; ufo 7) */
  uint8_t set_lut[16][4];             /* per bank sprite ((off - 50) / 10, explosions 8 + (off - 127) / 10): up to 4 candidate sets, 255 = none */
  uint32_t inv32[TBX_AREA_MAX_DST + 1]; /* ceil(2^32 / n) for n >= 2 */
  uint32_t plain[TBX_AREA_MAX_DST][4]; /* per output row: the output columns all of whose real taps are background in base frame 0 */
  /* THE SCORE AS ONE STRIP.  Its digits are 8 source pixels apart, so neighbouring digits feed a common output column and no
   * digit can be a patch of its own.  But an output column is fed by at most two neighbouring digit slots: sc_px holds every
   * pixel of the strip for every pair of digits (10 = no digit) in those two slots, resolved on the host from base frame 0 with
   * the digits drawn.  sc_ok == 0: the geometry does not allow it (the digits are then evaluated pixel by pixel). */
  int32_t sc_ok, sc_gray;
  int32_t sc_dx0, sc_ncol, sc_dy0, sc_nrow;            /* output pixels fed by the ten digit slots */
  uint8_t sc_slot[TBX_SC_MAX_COLS];                    /* per strip column: the lowest slot that feeds it (255: none) */
  uint8_t sc_px[TBX_SC_MAX_COLS][11][11][TBX_SC_MAX_ROWS]; /* [column][digit in that slot][digit in the next slot][row] */
} TbxSiDirect;
/* patch of set s at phase (x mod px_period, y mod py_period): patches[(s * py_period + yphase) * px_period + xphase] */

/* ------------------------------------------------------------------ Amidar: a grid of cells with four looks
 * The maze is 32 x 31 tiles of 4 x 5 pixels; a tile looks empty (background), unpainted, painted, or -- inside a painted box --
 * filled.  The horizontal sum of a tile row at an output column depends on the looks of at most two neighbouring tiles: a
 * 16-entry look-up per column, shared by all tile rows (they have the same geometry).  Only the output words x rows fed by a
 * tile whose look differs from the config board's are recomputed.  Enemies and player (6 x 7 rectangles) are evaluated like
 * Breakout's movers, their source windows built from the tile looks. */
#define AMI_N_MOVERS (TBX_AMI_MAX_ENEMIES + 1) /* enemies in index order, then the player (draw order) */
typedef struct TbxAmiDirect {
  int32_t ok;
  int32_t mdy0, mdy1;            /* output rows fed by the maze's source rows (inclusive) */
  int32_t hud_dylo;              /* first output row fed by a HUD digit row */
  uint32_t gray[4];              /* look -> gray: background, unpainted, painted, box fill */
  uint32_t player_gray, enemy_gray;
  uint32_t base_looks[TBX_AMI_BH][2]; /* the config board as 2-bit looks (what base frame 1 shows) */
  uint8_t xcol[TBX_AREA_MAX_SRC];     /* tile column of source column x, 255 = none */
  uint8_t yrow[TBX_AREA_MAX_SRC];     /* tile row of source row y, 255 = none */
  alignas(4) uint8_t col0[TBX_AREA_MAX_DST];     /* per output column: its taps touch tile columns col0 and col0 + 1 only */
  uint8_t ysel[TBX_AREA_MAX_DST][TBX_AREA_MAX_TAPS]; /* per output row and tap: tile row, 255 = a background row */
  uint32_t dyrows[TBX_AREA_MAX_DST];  /* per output row: mask of the tile rows its taps touch */
  uint32_t wordcols[32][2];           /* per output word: the tile columns that feed it, as a mask over the 2-bit look fields */
  uint32_t inv32[TBX_AREA_MAX_DST + 1];
  alignas(16) float hlut[16][TBX_AREA_MAX_DST]; /* [look(col0) | look(col0 + 1) << 2][dx] */
} TbxAmiDirect;

/* tile tags (2 bits each, 16 per word) -> looks: Empty 0, Unpainted / ChaseMarker 1, Painted 2 */
TBX_HD uint32_t ami_looks_of_tags(uint32_t t) {
  const uint32_t hi = (t >> 1) & 0x55555555u, lo = t & 0x55555555u, both = hi & lo;
  return ((hi | lo) & ~both) | (both << 1);
}

#endif
