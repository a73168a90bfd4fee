/* brk_img_check.cpp -- TEST-ONLY host build of the Breakout direct kernel's shared-memory image (tbx_direct.h,
 * tbx::build_brk_img), for tests/test_direct_image_cpu.py, which compiles it with the library's host half (tbx_host.cpp).
 * Not part of libtoybox_b200.so.
 */
#include "../../toybox_b200/csrc/tbx_host.h"
#include "../../toybox_b200/csrc/tbx_breakout.h"
#include "../../toybox_b200/csrc/tbx_direct.h"
#include <exception>
#include <memory>
#include <string.h>
#include <vector>

extern "C" {

/* The Breakout direct kernel's shared-memory image (tbx::build_brk_img) at out_w x out_h, for the default config (rows == 0) or
 * one with `rows` brick rows and other row colours, checked region by region against the tables it copies.  Returns -1 when
 * the direct kernel does not cover the pair, 0 when every region matches, else 1 + the first region that differs.  info (16):
 * TX, TY, nrows, n_static, the cached-digits flag, TBX_WORDS(BrkRec), then the region offsets in image order (flags, dig, rowcls,
 * inv, xdlo, xdhi, ydlo, ydhi, xcol, yrow, bgray, wordcols, col0, dyrows, hsel, base1, plan, hlut, hstatic, cls) and the
 * image's size: info[6 ..] (21 values, so info needs 27). */
int dc_brk_img(int out_w, int out_h, int rows, int32_t *info) {
  tbx::Config c;
  tbx::default_config(TBX_BREAKOUT, c);
  if (rows > 0) {
    const uint32_t cols[3] = {0xff2a48c8u, 0xff30a0b4u, 0xff10c020u};
    c.brk.n_rows = rows;
    for (int r = 0; r < rows; r++) c.brk.row_colors[r] = cols[r % 3] + (uint32_t)r * 0x050301u;
    tbx::brk_finish_cfg(c.brk);
  }
  BrkTable t;
  tbx::brk_default_table(c.brk, t);
  tbx::brk_mark_delta_ok(c, t);
  const int W = TBX_BRK_W, H = TBX_BRK_H;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &) { return -1; }
  if (!tbx::build_area_plan(rs, pl)) return -1;
  std::vector<uint32_t> rgba((size_t)W * H);
  std::vector<uint8_t> base0((size_t)W * H), base1((size_t)W * H), base1_out((size_t)out_w * out_h);
  tbx::build_base_frame(c, &t, 0, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base0.data());
  tbx::build_base_frame(c, &t, 1, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base1.data());
  tbx::area_resize(base1.data(), rs, base1_out.data());
  std::vector<TbxDigitPatch> patches((size_t)TBX_DP_SLOTS * 10);
  tbx::build_digit_patches(c, &t, rs, pl, base1.data(), patches.data());
  std::unique_ptr<TbxBrkDirect> A(new TbxBrkDirect);
  tbx::build_brk_direct(c, t, rs, pl, base0.data(), *A);
  if (!A->ok) return -1;
  /* the kernel instantiation the library launches for the plan (inst_taps, tbx_direct_launch.h) */
  const int tx = pl.tx <= 3 ? 3 : pl.tx <= 4 ? 4 : 5, ty = pl.ty <= 3 ? 3 : 4;
  std::vector<uint8_t> img;
  tbx::build_brk_img(*A, pl, tx, ty, base1_out.data(), patches.data(), img);
  const TbxBrkImgLayout L = brk_img_layout(tx, ty, out_w, out_h, A->nrows, A->n_static, A->n_cls);
  const int32_t offs[21] = {TBX_BI_FLAGS, TBX_BI_DIG, TBX_BI_ROWCLS, TBX_BI_INV, TBX_BI_XDLO, TBX_BI_XDHI, TBX_BI_YDLO, TBX_BI_YDHI,
                            TBX_BI_XCOL, TBX_BI_YROW, TBX_BI_BGRAY, TBX_BI_WORDCOLS, TBX_BI_COL0, TBX_BI_DYROWS, TBX_BI_HSEL, L.base1, L.plan, L.hlut,
                            L.hstatic, L.cls, L.bytes};
  info[0] = tx; info[1] = ty; info[2] = A->nrows; info[3] = A->n_static; info[5] = TBX_WORDS(BrkRec);
  for (int i = 0; i < 21; i++) info[6 + i] = offs[i];
  if ((size_t)L.bytes != img.size()) return 100;
  const uint8_t *b = img.data();
  int32_t flag;
  memcpy(&flag, b + TBX_BI_FLAGS, 4);
  info[4] = flag;
  /* the kernel's old per-CTA copy loops, restated: what each region must hold */
  bool fit = true;
  for (int e = 0; e < TBX_BRK_DIG_SLOTS * 10; e++) {
    const int cid = e / 10, slot = cid < 4 ? cid : cid + TBX_MAX_DIGITS - 4;
    const TbxDigitPatch &P = patches[slot * 10 + e % 10];
    fit &= P.w * P.h <= 48;
    if (memcmp(b + TBX_BI_DIG + 52 * e, &P, 52)) return 1 + 1;
  }
  if (flag != (fit ? 1 : 0)) return 1 + 0;
  if (memcmp(b + TBX_BI_ROWCLS, A->rowcls, H)) return 1 + 2;
  if (memcmp(b + TBX_BI_INV, A->inv32, 4 * (TBX_AREA_MAX_DST + 1))) return 1 + 3;
  if (memcmp(b + TBX_BI_XDLO, pl.xdlo, W)) return 1 + 4;
  if (memcmp(b + TBX_BI_XDHI, pl.xdhi, W)) return 1 + 5;
  if (memcmp(b + TBX_BI_YDLO, pl.ydlo, H)) return 1 + 6;
  if (memcmp(b + TBX_BI_YDHI, pl.ydhi, H)) return 1 + 7;
  if (memcmp(b + TBX_BI_XCOL, A->xcol, W)) return 1 + 8;
  if (memcmp(b + TBX_BI_YROW, A->yrow, H)) return 1 + 9;
  if (memcmp(b + TBX_BI_BGRAY, A->brickgray, TBX_BRK_MAX_BRICKS)) return 1 + 10;
  if (memcmp(b + TBX_BI_WORDCOLS, A->wordcols, 4 * 32)) return 1 + 11;
  if (memcmp(b + TBX_BI_COL0, A->col0, out_w)) return 1 + 12;
  if (memcmp(b + TBX_BI_DYROWS, A->dyrows, out_h)) return 1 + 13;
  for (int dy = 0; dy < out_h; dy++)
    for (int k = 0; k < ty; k++)
      if (b[TBX_BI_HSEL + dy * ty + k] != A->hsel[dy][k]) return 1 + 14;
  if (memcmp(b + L.base1, base1_out.data(), (size_t)out_w * out_h)) return 1 + 15;
  const int ps = brk_plan_pitch(out_w, out_h), hs = (out_w + 3) & ~3;
  for (int i = 0; i < ps; i++) {
    const int jx = i < out_w ? i : out_w - 1, jy = i < out_h ? i : out_h - 1;
    for (int k = 0; k < tx; k++) if (memcmp(b + L.plan + 4 * (k * ps + i), &pl.xalpha[k][jx], 4)) return 1 + 16;
    for (int k = 0; k < ty; k++) if (memcmp(b + L.plan + 4 * ((tx + k) * ps + i), &pl.yalpha[k][jy], 4)) return 1 + 16;
    if (memcmp(b + L.plan + 4 * (tx + ty) * ps + 2 * i, &pl.xs0[jx], 2) || memcmp(b + L.plan + 4 * (tx + ty) * ps + 2 * (ps + i), &pl.ys0[jy], 2)) return 1 + 16;
  }
  for (int r = 0; r < A->nrows; r++)
    for (int bits = 0; bits < 4; bits++)
      if (memcmp(b + L.hlut + 4 * (size_t)((r * 4 + bits) * hs), A->hlut[r][bits], 4 * (size_t)out_w)) return 1 + 17;
  for (int s = 0; s < A->n_static; s++)
    if (memcmp(b + L.hstatic + 4 * (size_t)(s * hs), A->hstatic[s], 4 * (size_t)out_w)) return 1 + 18;
  if (memcmp(b + L.cls, A->clsrows, (size_t)A->n_cls * W + 16)) return 1 + 19;
  return 0;
}

}
