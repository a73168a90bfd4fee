/* direct_check.cpp -- TEST-ONLY host build of two shortcuts of the Breakout direct kernel (tbx_direct.h,
 * tbx_render_direct.cuh), for tests/test_direct_digits_cpu.py, which compiles it with the library's host half
 * (tbx_host.cpp).  Default Breakout config throughout.  Not part of libtoybox_b200.so.
 */
#include "../../toybox_b200/csrc/tbx_host.h"
#include "../../toybox_b200/csrc/tbx_breakout.h"
#include "../../toybox_b200/csrc/tbx_direct.h"
#include <exception>
#include <vector>

extern "C" {

/* The Breakout movers of record `rec` both ways: out[10 (m + 1) .. + 4] = brk_mover (through the draw-list primitive),
 * out[10 (m + 1) + 5 .. + 9] = brk_mover_rec (straight from the record, what the direct kernel runs); x0, y0, x1, y1, gray
 * each, for m = -1 .. BRK_N_MOVERS (BRK_N_MOVERS + 2 rows). */
int dc_brk_movers(const uint32_t *rec, int32_t *out) {
  tbx::Config c;
  tbx::default_config(TBX_BREAKOUT, c);
  for (int m = -1; m <= BRK_N_MOVERS; m++) {
    const TbxMover a = brk_mover(rec, c.brk, 77u, 133u, m);
    const TbxMover b = brk_mover_rec(TbxAcc{const_cast<uint32_t *>(rec), 1}, 77u, 133u, m);
    int32_t *o = out + 10 * (m + 1);
    o[0] = a.x0; o[1] = a.y0; o[2] = a.x1; o[3] = a.y1; o[4] = (int32_t)a.gray;
    o[5] = b.x0; o[6] = b.y0; o[7] = b.x1; o[8] = b.y1; o[9] = (int32_t)b.gray;
  }
  return 0;
}

/* record word offsets of the mover fields: paddle_px, paddle_py, paddle_width, ball_radius, n_balls, ball[0] (x, y as f64 at
 * +0, +2; 8 words per ball) */
void dc_brk_mover_words(int32_t *out) {
  out[0] = BRK_W(paddle_px); out[1] = BRK_W(paddle_py); out[2] = BRK_W(paddle_width); out[3] = BRK_W(ball_radius); out[4] = BRK_W(n_balls); out[5] = BRK_W(ball);
}

/* The output rectangles of the HUD digit patches the library builds for out_w x out_h on base frame 1 (build_digit_patches):
 * out[4 (10 slot + digit) ..] = x0, y0, w, h (w == 0: no patch).  Returns the number of slots, -1 for a size the library
 * refuses. */
int dc_digit_patch_boxes(int out_w, int out_h, int32_t *out) {
  tbx::Config c;
  tbx::default_config(TBX_BREAKOUT, c);
  BrkTable t;
  tbx::brk_default_table(c.brk, t);
  tbx::brk_mark_delta_ok(c, t);
  const int W = TBX_BRK_W, H = TBX_BRK_H;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &) { return -1; }
  if (!tbx::build_area_plan(rs, pl)) return -1;
  std::vector<uint32_t> rgba((size_t)W * H);
  std::vector<uint8_t> base1((size_t)W * H);
  tbx::build_base_frame(c, &t, 1, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base1.data());
  std::vector<TbxDigitPatch> patches((size_t)TBX_DP_SLOTS * 10);
  tbx::build_digit_patches(c, &t, rs, pl, base1.data(), patches.data());
  for (int i = 0; i < TBX_DP_SLOTS * 10; i++) { out[4 * i] = patches[i].x0; out[4 * i + 1] = patches[i].y0; out[4 * i + 2] = patches[i].w; out[4 * i + 3] = patches[i].h; }
  return TBX_DP_SLOTS;
}

}
