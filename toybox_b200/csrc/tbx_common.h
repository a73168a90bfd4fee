/* tbx_common.h -- helpers shared by every game engine: exact-f64 ops, xoroshiro128+, the word-plane
 * accessor, ALE action decoding, colour/luma, the draw-list primitive.
 *
 * The engines in tbx_{breakout,space_invaders,amidar}.h are written once as TBX_HD inline functions
 * over an accessor.  nvcc compiles them into the sm_100a kernels (tbx_kernels.cu); tests/emu compiles
 * the very same functions for the host so the game logic can be checked against the oracle in the
 * CPU-only test tier.  The product library never contains or calls a host build of them.
 */
#ifndef TBX_COMMON_H
#define TBX_COMMON_H
#include "tbx_records.h"

#if defined(__CUDACC__)
#define TBX_HD __host__ __device__ __forceinline__
#define TBX_HDM __host__ __device__ __forceinline__
#else
#define TBX_HD static inline
#define TBX_HDM inline
#endif

/* ---- arithmetic, one IEEE-754 operation each, never contracted into FMA */
#if defined(__CUDA_ARCH__)
TBX_HD double tbx_dmul(double a, double b) { return __dmul_rn(a, b); }
TBX_HD double tbx_dadd(double a, double b) { return __dadd_rn(a, b); }
TBX_HD double tbx_dsub(double a, double b) { return __dsub_rn(a, b); }
TBX_HD double tbx_ddiv(double a, double b) { return __ddiv_rn(a, b); }
TBX_HD double tbx_dsqrt(double a) { return __dsqrt_rn(a); }
TBX_HD float tbx_fmul(float a, float b) { return __fmul_rn(a, b); }
TBX_HD float tbx_fadd(float a, float b) { return __fadd_rn(a, b); }
TBX_HD int tbx_f2i_rn(float v) { return __float2int_rn(v); } /* round half to even, as cvRound */
/* the same two conversions without the quarter-rate conversion pipe: exact u8 -> f32 through the 2^23 exponent
 * trick, and round-half-even f32 -> int for |v| < 2^22 through the 1.5 * 2^23 magic add */
TBX_HD float tbx_u8f(uint32_t b) { return __fadd_rn(__uint_as_float(0x4B000000u | b), -8388608.0f); }
TBX_HD int tbx_f2i_rn_small(float v) { return __float_as_int(__fadd_rn(v, 12582912.0f)) - 0x4B400000; }
TBX_HD int tbx_ffs(uint32_t m) { return __ffs((int)m); }
TBX_HD int tbx_popc(uint32_t m) { return __popc(m); }
TBX_HD uint32_t tbx_mulhi(uint32_t a, uint32_t b) { return __umulhi(a, b); }
#else
#include <math.h>
TBX_HD double tbx_dmul(double a, double b) { return a * b; } /* host builds use -ffp-contract=off */
TBX_HD double tbx_dadd(double a, double b) { return a + b; }
TBX_HD double tbx_dsub(double a, double b) { return a - b; }
TBX_HD double tbx_ddiv(double a, double b) { return a / b; }
TBX_HD double tbx_dsqrt(double a) { return sqrt(a); }
TBX_HD float tbx_fmul(float a, float b) { return a * b; }
TBX_HD float tbx_fadd(float a, float b) { return a + b; }
TBX_HD int tbx_f2i_rn(float v) { return (int)lrintf(v); }
TBX_HD float tbx_u8f(uint32_t b) { return (float)b; }
TBX_HD int tbx_f2i_rn_small(float v) { return (int)lrintf(v); }
TBX_HD int tbx_ffs(uint32_t m) { return __builtin_ffs((int)m); }
TBX_HD int tbx_popc(uint32_t m) { return __builtin_popcount(m); }
TBX_HD uint32_t tbx_mulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
#endif

/* Rust `f64 as i32` as the engines use it: truncate, saturate, NaN -> 0 */
TBX_HD int tbx_d2i(double v) {
  if (!(v == v)) return 0;
  if (v >= 536870912.0) return 536870912;
  if (v <= -536870912.0) return -536870912;
  return (int)v;
}

/* ---- word-plane accessor: p points at word 0 of one env, consecutive words are `stride` apart.
 * stride = n_pad for the device planes, 1 for an AoS record (shared-memory staging, host records). */
struct TbxAcc {
  uint32_t *p;
  size_t stride;
  TBX_HDM uint32_t ld(int w) const { return p[(size_t)w * stride]; }
  TBX_HDM void st(int w, uint32_t v) const { p[(size_t)w * stride] = v; }
  TBX_HDM int32_t ldi(int w) const { return (int32_t)ld(w); }
  TBX_HDM void sti(int w, int32_t v) const { st(w, (uint32_t)v); }
  TBX_HDM uint64_t ld64(int w) const { return (uint64_t)ld(w) | ((uint64_t)ld(w + 1) << 32); }
  TBX_HDM void st64(int w, uint64_t v) const { st(w, (uint32_t)v); st(w + 1, (uint32_t)(v >> 32)); }
  TBX_HDM double ldd(int w) const {
    union { uint64_t u; double d; } c; c.u = ld64(w); return c.d;
  }
  TBX_HDM void std_(int w, double v) const {
    union { uint64_t u; double d; } c; c.d = v; st64(w, c.u);
  }
};

/* ---- xoroshiro128+ (55,14,36); pinned by the fixtures, SURVEY App. A.1 */
struct TbxRng { uint64_t s0, s1; };
TBX_HD uint64_t tbx_rotl64(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
TBX_HD uint64_t tbx_rng_next_u64(TbxRng &g) {
  uint64_t s0 = g.s0, s1 = g.s1, r = s0 + s1;
  s1 ^= s0;
  g.s0 = tbx_rotl64(s0, 55) ^ s1 ^ (s1 << 14);
  g.s1 = tbx_rotl64(s1, 36);
  return r;
}
TBX_HD uint32_t tbx_rng_next_u32(TbxRng &g) { return (uint32_t)(tbx_rng_next_u64(g) >> 32); }
/* uniform index in [0,n): widening multiply with a rejection zone (pinned by the Breakout fixture's
 * two-draw ball-start choice, SURVEY App. A.3) */
TBX_HD uint32_t tbx_rng_index(TbxRng &g, uint32_t n) {
  if (n == 0) return 0;
  int lz = 0;
  while (!((n << lz) & 0x80000000u)) lz++;
  uint32_t zone = (n << lz) - 1u;
  for (;;) {
    uint64_t m = (uint64_t)tbx_rng_next_u32(g) * (uint64_t)n;
    if ((uint32_t)m <= zone) return (uint32_t)(m >> 32);
  }
}
TBX_HD double tbx_rng_f64(TbxRng &g) { return (double)(tbx_rng_next_u64(g) >> 11) * (1.0 / 9007199254740992.0); }
TBX_HD void tbx_rng_seed(TbxRng &g, uint32_t seed) {
  g.s0 = 0x193a6754a8a7d469ULL ^ (uint64_t)seed;
  g.s1 = 0x97830e05113ba7bbULL;
}
TBX_HD TbxRng tbx_rng_load(const TbxAcc &S, int w) { TbxRng g; g.s0 = S.ld64(w); g.s1 = S.ld64(w + 2); return g; }
TBX_HD void tbx_rng_store(const TbxAcc &S, int w, const TbxRng &g) { S.st64(w, g.s0); S.st64(w + 2, g.s1); }

#define TBX_HW(field) TBX_W(TbxHdr, field)

/* ---- ALE action id -> Input bitmask, toybox/envs/atari/constants.py:16-35; -1 = invalid id */
TBX_HD int tbx_ale_action_to_input(int a) {
  if (a < 0 || a > 17) return -1;
  int m = 0;
  /* 0 NOOP 1 FIRE 2 UP 3 RIGHT 4 LEFT 5 DOWN 6 UR 7 UL 8 DR 9 DL 10 UF 11 RF 12 LF 13 DF 14 URF 15 ULF 16 DRF 17 DLF */
  const uint32_t up = 0x0C4C4u, right = 0x14948u, left = 0x29290u, down = 0x32320u, fire = 0x3FC02u;
  if ((up >> a) & 1u) m |= TBX_IN_UP;
  if ((right >> a) & 1u) m |= TBX_IN_RIGHT;
  if ((left >> a) & 1u) m |= TBX_IN_LEFT;
  if ((down >> a) & 1u) m |= TBX_IN_DOWN;
  if ((fire >> a) & 1u) m |= TBX_IN_BUTTON1;
  return m;
}

/* ---- counter-based draws: the splitmix64 finaliser of (seed, env, t) */
TBX_HD uint64_t tbx_mix(uint64_t seed, uint64_t env, uint64_t t) {
  uint64_t z = seed + env * 0x9E3779B97F4A7C15ULL + t * 0xD1B54A32D192ED03ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
/* synthetic action stream of the bench / parity tests (SURVEY 8d), and the no-op counts of the wrapper stack: uniform over n_legal */
TBX_HD uint32_t tbx_action_index(uint64_t seed, uint64_t env, uint64_t t, uint32_t n_legal) {
  return (uint32_t)(((tbx_mix(seed, env, t) >> 32) * (uint64_t)n_legal) >> 32);
}
/* the sticky-action draw of env `env` on its frame `f` (tbx_wrap.cuh): uniform over [0, 2^32).  The salt separates this stream
 * from the no-op stream when both use one seed. */
#define TBX_STICKY_SALT 0x5354494B59414354ULL /* "STIKYACT" */
TBX_HD uint32_t tbx_sticky_draw(uint64_t seed, uint64_t env, uint64_t f) { return (uint32_t)(tbx_mix(seed ^ TBX_STICKY_SALT, env, f) >> 32); }

/* ---- colour: r | g<<8 | b<<16 | a<<24 (the byte order of an RGBA pixel in memory) */
TBX_HD uint32_t tbx_rgba(uint32_t r, uint32_t g, uint32_t b, uint32_t a) { return r | (g << 8) | (b << 16) | (a << 24); }
/* grayscale byte of a colour: (0.299 r + 0.587 g + 0.114 b) truncated, evaluated in f64 */
TBX_HD uint32_t tbx_luma(uint32_t c) {
  double r = (double)(c & 255u), g = (double)((c >> 8) & 255u), b = (double)((c >> 16) & 255u);
  double v = tbx_dadd(tbx_dadd(tbx_dmul(0.299, r), tbx_dmul(0.587, g)), tbx_dmul(0.114, b));
  return (uint32_t)(int)v & 255u;
}

/* ---- env-level bookkeeping of ToyboxBaseEnv.step (toybox/envs/atari/base.py:136-147), run after the
 * game transition: reward = max(score - prev_score, 0), done = lives <= 0, episode counters. */
struct TbxStepOut { int reward, done, score, lives, ep_len, ep_return, episode_ended; };
TBX_HD TbxStepOut tbx_bookkeep(const TbxAcc &S, int lives_before) {
  TbxStepOut o;
  o.score = S.ldi(TBX_HW(score)); o.lives = S.ldi(TBX_HW(lives));
  int r = o.score - S.ldi(TBX_HW(prev_score));
  o.reward = r < 0 ? 0 : r;
  o.done = o.lives <= 0;
  o.ep_len = S.ldi(TBX_HW(ep_len)) + 1;
  o.ep_return = S.ldi(TBX_HW(ep_return)) + o.reward;
  o.episode_ended = o.done && lives_before > 0;
  S.sti(TBX_HW(prev_score), o.score);
  S.sti(TBX_HW(ep_len), o.ep_len);
  S.sti(TBX_HW(ep_return), o.ep_return);
  return o;
}

/* ---- INTER_AREA arithmetic (general path of cv2.resize), f32, taps accumulated in table order.
 * horizontal: one source row -> buf[dx]; vertical: buf rows -> rounded (half to even), saturated byte. */
TBX_HD float tbx_area_h(const uint8_t *row, const TbxResizeAxis &ax, int dx) {
  int k = ax.start[dx], k1 = ax.start[dx + 1];
  float acc = tbx_fmul((float)row[ax.si[k]], ax.alpha[k]);
  for (k++; k < k1; k++) acc = tbx_fadd(acc, tbx_fmul((float)row[ax.si[k]], ax.alpha[k]));
  return acc;
}
/* buf holds source rows starting at row ys0, `stride` floats per row */
TBX_HD uint8_t tbx_area_v(const float *buf, int stride, int ys0, const TbxResizeAxis &ay, int dy, int dx) {
  int k = ay.start[dy], k1 = ay.start[dy + 1];
  float s = tbx_fmul(ay.alpha[k], buf[(ay.si[k] - ys0) * stride + dx]);
  for (k++; k < k1; k++) s = tbx_fadd(s, tbx_fmul(ay.alpha[k], buf[(ay.si[k] - ys0) * stride + dx]));
  int v = tbx_f2i_rn(s);
  return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
}

/* ---- draw-list groups: consecutive slot ranges painted one after the other.  Inside a PARALLEL group no two
 * primitives can conflict (disjoint rectangles, or one colour), so they may be painted in any order; a SERIAL
 * group is painted strictly in slot order. */
enum { TBX_GROUP_PARALLEL = 0, TBX_GROUP_SERIAL = 1, TBX_GROUP_NOSYNC = 2 /* flag: provably disjoint from the next group */ };

/* ---- draw-list primitive (16 bytes): a rectangle, optionally masked by a 1-bit sprite.
 * Pixel (px,py) of the rectangle is painted iff bw == 0 or bit (bw-1 - px/sx) of rows[py/sy] is set,
 * rows = sprite bank + off, or (off & TBX_PRIM_STATE) the env's own record words + (off & 0x7fff). */
#define TBX_PRIM_STATE 0x8000u
struct TbxPrim {
  int16_t x, y, w, h; /* h == 0: empty slot */
  uint32_t color;     /* RGBA */
  uint16_t off;
  uint8_t bw, scale;  /* scale = sx | sy << 4 */
};
TBX_HD TbxPrim tbx_prim_none() { TbxPrim p; p.x = p.y = p.w = p.h = 0; p.color = 0; p.off = 0; p.bw = 0; p.scale = 0x11; return p; }
TBX_HD TbxPrim tbx_prim_rect(uint32_t color, int x, int y, int w, int h) {
  TbxPrim p = tbx_prim_none();
  if (w <= 0 || h <= 0) return p;
  /* far-away coordinates are clipped to 16 bits; the painter clips to the canvas anyway */
  long long xe = (long long)x + w, ye = (long long)y + h;
  int x0 = x < -30000 ? -30000 : x > 30000 ? 30000 : x, y0 = y < -30000 ? -30000 : y > 30000 ? 30000 : y;
  int x1 = xe > 30000 ? 30000 : xe < -30000 ? -30000 : (int)xe;
  int y1 = ye > 30000 ? 30000 : ye < -30000 ? -30000 : (int)ye;
  if (x1 <= x0 || y1 <= y0) return p;
  p.x = (int16_t)x0; p.y = (int16_t)y0; p.w = (int16_t)(x1 - x0); p.h = (int16_t)(y1 - y0); p.color = color;
  return p;
}
TBX_HD TbxPrim tbx_prim_sprite(uint32_t color, int x, int y, int bw, int bh, uint32_t off, int sx, int sy) {
  TbxPrim p = tbx_prim_none();
  if (x < -30000 || x > 30000 || y < -30000 || y > 30000) return p; /* entirely off any canvas */
  p.x = (int16_t)x; p.y = (int16_t)y; p.w = (int16_t)(bw * sx); p.h = (int16_t)(bh * sy); p.color = color;
  p.off = (uint16_t)off; p.bw = (uint8_t)bw; p.scale = (uint8_t)(sx | (sy << 4));
  return p;
}
/* does the primitive paint canvas pixel (cx,cy)?  (reference painter used by the CPU-tier emulation and
 * by small device paths; the kernels' band painter walks spans instead) */
TBX_HD bool tbx_prim_covers(const TbxPrim &p, const uint32_t *bank, const uint32_t *rec, int cx, int cy) {
  int px = cx - p.x, py = cy - p.y;
  if (px < 0 || py < 0 || px >= p.w || py >= p.h) return false;
  if (p.bw == 0) return true;
  const uint32_t *rows = (p.off & TBX_PRIM_STATE) ? rec + (p.off & 0x7fffu) : bank + p.off;
  int sx = p.scale & 15, sy = p.scale >> 4;
  return (rows[py / sy] >> (p.bw - 1 - px / sx)) & 1u;
}

/* ---- sprite bank (word offsets).  Font: 3x5 digits; the rest are the Space Invaders sprites. */
#define TBX_BANK_FONT 0      /* [10][5] */
#define TBX_BANK_INVADER 50  /* [3 kinds][2 poses][10] */
#define TBX_BANK_SHIP 110    /* [10] */
#define TBX_BANK_UFO 120     /* [7] */
#define TBX_BANK_BOOM 127    /* [2][10] */
#define TBX_BANK_WORDS 147
#define TBX_BANK_INIT { \
  7, 5, 5, 5, 7,  2, 6, 2, 2, 7,  7, 1, 7, 4, 7,  7, 1, 7, 1, 7,  5, 5, 7, 1, 1, \
  7, 4, 7, 1, 7,  7, 4, 7, 5, 7,  7, 1, 1, 1, 1,  7, 5, 7, 5, 7,  7, 5, 7, 1, 7, \
  0x0810, 0x0420, 0x0FF0, 0x1BD8, 0x3FFC, 0x2FF4, 0x2814, 0x0660, 0, 0, \
  0x0810, 0x2424, 0x2FF4, 0x3BDC, 0x3FFC, 0x1FF8, 0x0810, 0x1008, 0, 0, \
  0x0180, 0x03C0, 0x07E0, 0x0DB0, 0x0FF0, 0x0240, 0x05A0, 0x0A50, 0, 0, \
  0x0180, 0x03C0, 0x07E0, 0x0DB0, 0x0FF0, 0x05A0, 0x0810, 0x0420, 0, 0, \
  0x03C0, 0x1FF8, 0x3FFC, 0x39CC, 0x3FFC, 0x0660, 0x0DB0, 0x300C, 0, 0, \
  0x03C0, 0x1FF8, 0x3FFC, 0x39CC, 0x3FFC, 0x0E70, 0x1998, 0x0C30, 0, 0, \
  0x0100, 0x0380, 0x0380, 0x3FF8, 0x7FFC, 0x7FFC, 0x7FFC, 0x7FFC, 0x7FFC, 0x7FFC, \
  0x07E0, 0x1FF8, 0x3FFC, 0x6DB6, 0xFFFF, 0x399C, 0x1008, \
  0x0890, 0x4512, 0x2244, 0x1008, 0xC003, 0x1008, 0x2244, 0x4512, 0x0890, 0x0000, \
  0x1248, 0x0420, 0x4812, 0x2004, 0x0240, 0x9009, 0x0420, 0x2814, 0x4002, 0x1248 }

/* right-aligned decimal digits as sprite prims: slot k (0 = least significant) of at most `max_digits`;
 * mirrors the HUD digit layout of the draw lists (3x5 font, 1 column gap) */
TBX_HD TbxPrim tbx_prim_digit(uint32_t color, int x_right, int y, int value, int sx, int sy, int k) {
  const uint32_t v = value < 0 ? 0u : (uint32_t)value;
  uint32_t q; /* v / 10^k with compile-time divisors (multiply-shift, no division unit) */
  switch (k) {
    case 0: q = v; break;
    case 1: q = v / 10u; break;
    case 2: q = v / 100u; break;
    case 3: q = v / 1000u; break;
    case 4: q = v / 10000u; break;
    case 5: q = v / 100000u; break;
    case 6: q = v / 1000000u; break;
    case 7: q = v / 10000000u; break;
    case 8: q = v / 100000000u; break;
    default: q = v / 1000000000u; break;
  }
  if (k > 0 && q == 0) return tbx_prim_none();
  return tbx_prim_sprite(color, x_right - 3 * sx - 4 * sx * k, y, 3, 5, TBX_BANK_FONT + 5 * (q % 10u), sx, sy);
}
#define TBX_MAX_DIGITS 10

#endif
