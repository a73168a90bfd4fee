/* emu.cpp -- TEST-ONLY host build of the engine headers (tbx_breakout.h, tbx_space_invaders.h,
 * tbx_amidar.h) plus the library's host half (tbx_host.cpp), so the CPU-only test tier can check the
 * very functions the CUDA kernels are compiled from -- transition, new_game, draw list, INTER_AREA
 * arithmetic, JSON codecs -- against the oracle without a GPU.  It is NOT part of libtoybox_b200.so and the
 * product never loads it: the product path has no CPU fallback.
 *
 * One `Emu` is one environment (an AoS record, stride 1).  Painting uses a plain sequential painter's
 * algorithm over the draw list; the kernels' warp-band painter is checked on the GPU tier.
 */
#include "../../toybox_b200/csrc/tbx_host.h"
#include "../../toybox_b200/csrc/tbx_breakout.h"
#include "../../toybox_b200/csrc/tbx_space_invaders.h"
#include "../../toybox_b200/csrc/tbx_amidar.h"
#include "../../toybox_b200/csrc/tbx_direct.h"
#include <string.h>
#include <stdlib.h>
#include <memory>
#include <string>
#include <vector>

using tbxjson::Value;

static const uint32_t BANK[TBX_BANK_WORDS] = TBX_BANK_INIT;
static thread_local std::string g_err;

struct Emu {
  int game;
  const tbx::GameInfo *info;
  tbx::Config cfg;
  std::vector<BrkTable> brk_tables;
  std::vector<AmiTable> ami_tables;
  std::vector<uint32_t> rec;
  TbxAcc acc() { TbxAcc S; S.p = rec.data(); S.stride = 1; return S; }
};
template <class TT> static int intern(std::vector<TT> &v, const TT &t) {
  for (size_t i = 0; i < v.size(); i++) if (memcmp(&v[i], &t, sizeof t) == 0) return (int)i;
  v.push_back(t);
  return (int)v.size() - 1;
}
static void install_default_table(Emu *e) {
  if (e->game == TBX_BREAKOUT) { BrkTable t; tbx::brk_default_table(e->cfg.brk, t); tbx::brk_mark_delta_ok(e->cfg, t); e->cfg.brk.default_tbl = intern(e->brk_tables, t); }
  else if (e->game == TBX_AMIDAR) { AmiTable t; tbx::ami_default_table(e->cfg.ami, t); e->cfg.ami.default_tbl = intern(e->ami_tables, t); }
}
static void new_game(Emu *e) {
  TbxAcc S = e->acc();
  if (e->game == TBX_BREAKOUT) brk_new_game(S, e->cfg.brk);
  else if (e->game == TBX_AMIDAR) ami_new_game(S, e->cfg.ami, e->ami_tables.data());
  else si_new_game(S, e->cfg.si);
}
static char *dup_str(const std::string &s) { char *o = (char *)malloc(s.size() + 1); memcpy(o, s.c_str(), s.size() + 1); return o; }

extern "C" {

const char *emu_last_error(void) { return g_err.c_str(); }
void emu_free_str(char *s) { free(s); }

Emu *emu_create(const char *game, const char *cfg_json) {
  int g = tbx::game_from_name(game);
  if (g < 0) { g_err = "unknown game"; return 0; }
  Emu *e = new Emu();
  e->game = g; e->info = tbx::game_info(g);
  try {
    tbx::default_config(g, e->cfg);
    if (cfg_json) tbx::config_from_json(e->cfg, tbxjson::parse(cfg_json));
    install_default_table(e);
  } catch (const std::exception &ex) { g_err = ex.what(); delete e; return 0; }
  e->rec.assign(e->info->rec_words, 0);
  const uint64_t *rand = g == TBX_BREAKOUT ? e->cfg.brk.rand : g == TBX_AMIDAR ? e->cfg.ami.rand : e->cfg.si.rand;
  TbxAcc S = e->acc();
  S.st64(TBX_HW(sim_rand), rand[0]); S.st64(TBX_HW(sim_rand) + 2, rand[1]);
  for (int k = 0; k < e->info->new_games_at_ctor; k++) new_game(e);
  return e;
}
void emu_destroy(Emu *e) { delete e; }
int emu_rec_words(Emu *e) { return e->info->rec_words; }
uint32_t *emu_record(Emu *e) { return e->rec.data(); }
void emu_seed(Emu *e, uint32_t seed) {
  TbxRng g; tbx_rng_seed(g, seed);
  TbxAcc S = e->acc();
  S.st64(TBX_HW(sim_rand), g.s0); S.st64(TBX_HW(sim_rand) + 2, g.s1);
}
void emu_new_game(Emu *e) { new_game(e); }

/* the same sequence step_kernel runs for one env; returns -1 for an invalid ALE id */
int emu_step(Emu *e, int ale_action, int input_mask, int auto_reset, int32_t *out4) {
  TbxAcc S = e->acc();
  int in = input_mask >= 0 ? input_mask : tbx_ale_action_to_input(ale_action);
  int lives_before = S.ldi(TBX_HW(lives));
  if (in >= 0) {
    if (e->game == TBX_BREAKOUT) brk_step(S, e->cfg.brk, e->brk_tables.data(), in);
    else if (e->game == TBX_AMIDAR) ami_step(S, e->cfg.ami, e->ami_tables.data(), in);
    else si_step(S, e->cfg.si, in);
  }
  TbxStepOut o = tbx_bookkeep(S, lives_before);
  if (out4) { out4[0] = o.reward; out4[1] = o.done; out4[2] = o.score; out4[3] = o.lives; }
  if (o.done && auto_reset) new_game(e);
  return in < 0 ? -1 : 0;
}

static TbxPrim get_prim(Emu *e, int slot) {
  if (e->game == TBX_BREAKOUT) return brk_prim(e->rec.data(), e->cfg.brk, e->brk_tables.data(), slot);
  if (e->game == TBX_AMIDAR) return ami_prim(e->rec.data(), e->cfg.ami, e->ami_tables.data(), slot);
  return si_prim(e->rec.data(), slot);
}
/* mode: 0 rgba 1 rgb 2 gray 3 gray + INTER_AREA to out_w x out_h */
int emu_render(Emu *e, int mode, int out_w, int out_h, uint8_t *out) {
  const int W = e->info->width, H = e->info->height;
  uint32_t clearv = e->game == TBX_BREAKOUT ? e->cfg.brk.bg_color : e->game == TBX_AMIDAR ? e->cfg.ami.bg_color : SI_COLOR_BLACK;
  std::vector<uint32_t> canvas((size_t)W * H, clearv);
  for (int s = 0; s < e->info->n_slots; s++) {
    TbxPrim p = get_prim(e, s);
    if (p.h <= 0) continue;
    for (int y = p.y < 0 ? 0 : p.y; y < p.y + p.h && y < H; y++)
      for (int x = p.x < 0 ? 0 : p.x; x < p.x + p.w && x < W; x++)
        if (tbx_prim_covers(p, BANK, e->rec.data(), x, y)) canvas[(size_t)y * W + x] = p.color;
  }
  if (mode == 0) { memcpy(out, canvas.data(), (size_t)W * H * 4); return 0; }
  if (mode == 1) { for (int i = 0; i < W * H; i++) { out[3 * i] = canvas[i] & 255; out[3 * i + 1] = (canvas[i] >> 8) & 255; out[3 * i + 2] = (canvas[i] >> 16) & 255; } return 0; }
  std::vector<uint8_t> gray((size_t)W * H);
  for (int i = 0; i < W * H; i++) gray[i] = (uint8_t)tbx_luma(canvas[i]);
  if (mode == 2) { memcpy(out, gray.data(), gray.size()); return 0; }
  tbx::ResizeTab rs;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  std::vector<float> buf((size_t)H * out_w);
  for (int y = 0; y < H; y++) for (int dx = 0; dx < out_w; dx++) buf[(size_t)y * out_w + dx] = tbx_area_h(gray.data() + (size_t)y * W, rs.x, dx);
  for (int dy = 0; dy < out_h; dy++) for (int dx = 0; dx < out_w; dx++) out[dy * out_w + dx] = tbx_area_v(buf.data(), out_w, 0, rs.y, dy, dx);
  return 0;
}

/* The fused kernel's INTER_AREA algorithm, step for step on the host: static base frame + its pre-computed
 * down-sample, dynamic groups painted over the base, dirty rectangles (group bounding boxes / per-primitive
 * boxes of the in-order group), and only the output pixels fed by a dirty rectangle recomputed with the
 * zero-padded fixed-tap arithmetic of TbxAreaPlan.  Must equal emu_render(mode 3). */
int emu_render_fast(Emu *e, int out_w, int out_h, uint8_t *out) {
  const int W = e->info->width, H = e->info->height;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  if (!tbx::build_area_plan(rs, pl)) { g_err = "size pair outside the fused kernel's limits"; return -1; }
  const int base_id = e->game == TBX_BREAKOUT ? brk_base_id(e->rec.data(), e->cfg.brk, e->brk_tables.data())
                      : e->game == TBX_AMIDAR ? ami_base_id(e->rec.data(), e->cfg.ami, e->ami_tables.data()) : 0;
  std::vector<uint32_t> base((size_t)W * H);
  tbx::build_base_frame(e->cfg, e->game == TBX_BREAKOUT ? &e->brk_tables[e->cfg.brk.default_tbl] : 0, base_id, base.data());
  std::vector<uint8_t> canvas((size_t)W * H + 8 * W + 16, 0);
  tbx::frame_to_gray(base.data(), W * H, canvas.data());
  tbx::area_resize(canvas.data(), rs, out);
  struct Rect { int x0, y0, x1, y1; };
  std::vector<Rect> rects;
  const int ng = e->game == TBX_BREAKOUT ? BRK_N_GROUPS : e->game == TBX_AMIDAR ? AMI_N_GROUPS : SI_N_GROUPS;
  int covered = tbx::n_static_slots(e->game);
  for (int g = 0; g < ng; g++) {
    int gb, ge, mode;
    if (e->game == TBX_BREAKOUT) brk_group(g, e->rec.data(), e->brk_tables.data(), base_id, gb, ge, mode);
    else if (e->game == TBX_AMIDAR) ami_group(g, gb, ge, mode);
    else si_group(g, gb, ge, mode);
    if (gb != covered && gb < ge) { g_err = "groups do not tile the dynamic slots"; return -1; }
    if (gb >= ge) { covered = e->game == TBX_BREAKOUT && g == 1 ? BRK_SLOT_PADDLE : covered; continue; } /* skipped group */
    covered = ge;
    Rect box = {32767, 32767, -1, -1};
    const bool per_prim = (mode & TBX_GROUP_SERIAL) && ge - gb <= 32;
    for (int s = gb; s < ge; s++) {
      TbxPrim p = e->game == TBX_BREAKOUT ? brk_prim_delta(e->rec.data(), e->cfg.brk, e->brk_tables.data(), s, base_id)
                  : e->game == TBX_AMIDAR ? ami_prim_delta(e->rec.data(), e->cfg.ami, e->ami_tables.data(), s, base_id) : si_prim(e->rec.data(), s);
      Rect c = {p.x < 0 ? 0 : p.x, p.y < 0 ? 0 : p.y, p.x + p.w > W ? W : p.x + p.w, p.y + p.h > H ? H : p.y + p.h};
      if (p.h <= 0 || c.x0 >= c.x1 || c.y0 >= c.y1) continue;
      uint8_t val = (uint8_t)tbx_luma(p.color);
      for (int y = c.y0; y < c.y1; y++)
        for (int x = c.x0; x < c.x1; x++)
          if (tbx_prim_covers(p, BANK, e->rec.data(), x, y)) canvas[(size_t)y * W + x] = val;
      if (per_prim) rects.push_back(c);
      else { if (c.x0 < box.x0) box.x0 = c.x0; if (c.y0 < box.y0) box.y0 = c.y0; if (c.x1 > box.x1) box.x1 = c.x1; if (c.y1 > box.y1) box.y1 = c.y1; }
    }
    if (!per_prim && box.x1 > box.x0) rects.push_back(box);
  }
  if (covered != e->info->n_slots) { g_err = "groups do not tile the dynamic slots"; return -1; }
  for (size_t r = 0; r < rects.size(); r++) {
    const Rect &rc = rects[r];
    const int dx0 = pl.xdlo[rc.x0], dx1 = pl.xdhi[rc.x1 - 1], dy0 = pl.ydlo[rc.y0], dy1 = pl.ydhi[rc.y1 - 1];
    for (int dy = dy0; dy <= dy1; dy++)
      for (int dx = dx0; dx <= dx1; dx++) {
        const uint8_t *src = canvas.data() + (size_t)pl.ys0[dy] * W + pl.xs0[dx];
        float v = 0.0f;
        for (int k = 0; k < TBX_AREA_MAX_TAPS; k++) { /* zero-padded taps, as the kernel's fixed TY */
          const uint8_t *row = src + (size_t)k * W;
          float h = tbx_fmul((float)row[0], pl.xalpha[0][dx]);
          for (int t = 1; t < TBX_AREA_MAX_TAPS; t++) h = tbx_fadd(h, tbx_fmul((float)row[t], pl.xalpha[t][dx])); /* zero-padded taps */
          const float bh = tbx_fmul(pl.yalpha[k][dy], h);
          v = k == 0 ? bh : tbx_fadd(v, bh);
        }
        const int iv = tbx_f2i_rn(v);
        out[dy * out_w + dx] = (uint8_t)(iv < 0 ? 0 : iv > 255 ? 255 : iv);
      }
  }
  return 0;
}

/* The DIRECT INTER_AREA algorithm (tbx_direct.h, tbx_render_direct.cuh) on the host, phase by phase as the kernel runs
 * it: base down-sample, wall rows from the look-up tables (only the output words / rows a dead brick feeds), HUD digit
 * patches, then the movers' footprints evaluated tap by tap.  Returns 1 when the env is one the kernel hands to the
 * general tile kernel (not rendered here), 0 when `out` holds the frame; must then equal emu_render(mode 3). */
int emu_render_direct(Emu *e, int out_w, int out_h, uint8_t *out) {
  const int W = e->info->width, H = e->info->height;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  if (!tbx::build_area_plan(rs, pl)) { g_err = "size pair outside the fused kernel's limits"; return -1; }
  if (e->game != TBX_BREAKOUT) return 1;
  const BrkTable &dt = e->brk_tables[e->cfg.brk.default_tbl];
  std::vector<uint32_t> rgba((size_t)W * H);
  std::vector<uint8_t> base0((size_t)W * H), base1((size_t)W * H);
  tbx::build_base_frame(e->cfg, &dt, 0, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base0.data());
  tbx::build_base_frame(e->cfg, &dt, 1, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base1.data());
  static TbxBrkDirect A;
  tbx::build_brk_direct(e->cfg, dt, rs, pl, base0.data(), A);
  const uint32_t *R = e->rec.data();
  if (!A.ok || (int32_t)R[TBX_HW(tbl)] != e->cfg.brk.default_tbl) return 1;
  for (int y = 0; y < H && A.n_cls > 0; y++) /* base frame 0 by row classes: what the kernel's mover windows read */
    if (A.rowcls[y] >= A.n_cls || memcmp(A.clsrows + (size_t)A.rowcls[y] * W, base0.data() + (size_t)y * W, W) != 0) { g_err = "row class table differs from base frame 0"; return -1; }
  std::vector<TbxDigitPatch> patches((size_t)TBX_DP_SLOTS * 10);
  tbx::build_digit_patches(e->cfg, &dt, rs, pl, base1.data(), patches.data());
  TbxMover mv[BRK_N_MOVERS];
  int fx0[BRK_N_MOVERS], fx1[BRK_N_MOVERS], fy0[BRK_N_MOVERS], fy1[BRK_N_MOVERS];
  for (int m = 0; m < BRK_N_MOVERS; m++) {
    mv[m] = brk_mover(R, e->cfg.brk, A.paddle_gray, A.ball_gray, m);
    if (mv[m].x0 >= mv[m].x1) continue;
    fx0[m] = pl.xdlo[mv[m].x0]; fx1[m] = pl.xdhi[mv[m].x1 - 1]; fy0[m] = pl.ydlo[mv[m].y0]; fy1[m] = pl.ydhi[mv[m].y1 - 1];
    if (fy0[m] <= A.hud_dyhi) return 1;
  }
  const int32_t fields[2] = {(int32_t)R[TBX_HW(score)], (int32_t)R[TBX_HW(lives)]};
  for (int f = 0; f < 2; f++)
    for (int k = 0; k < TBX_MAX_DIGITS; k++) {
      const int d = tbx_digit_at(fields[f], k);
      if (d >= 0 && patches[(f * 10 + k) * 10 + d].w == 0) return 1;
    }
  tbx::area_resize(base1.data(), rs, out);
  /* wall */
  const uint32_t *alive = R + BRK_W(alive);
  const uint32_t full = (1u << A.nrows) - 1u;
  uint32_t deadcols = 0, deadrows = 0, rowmask[TBX_BRK_MAX_ROWS] = {0};
  for (int c = 0; c < A.ncols; c++) {
    const uint32_t v = brk_col_bits(alive, A.nrows, c);
    if (v != full) deadcols |= 1u << c;
    deadrows |= ~v & full;
    for (int r = 0; r < A.nrows; r++) rowmask[r] |= ((v >> r) & 1u) << c;
  }
  if (deadcols) {
    std::vector<float> hd((size_t)A.nrows * out_w);
    for (int r = 0; r < A.nrows; r++) for (int dx = 0; dx < out_w; dx++) hd[(size_t)r * out_w + dx] = brk_direct_h(A, r, rowmask[r], dx);
    int rlo = -1, rhi = -1;
    for (int dy = A.wdy0; dy <= A.wdy1; dy++) if (A.dyrows[dy] & deadrows) { if (rlo < 0) rlo = dy; rhi = dy; }
    for (int dy = rlo; rlo >= 0 && dy <= rhi; dy++)
      for (int w = 0; w < out_w / 4; w++) {
        if (!(A.wordcols[w] & deadcols)) continue;
        for (int dx = 4 * w; dx < 4 * w + 4; dx++) out[dy * out_w + dx] = brk_direct_wall_pixel<TBX_AREA_MAX_TAPS>(A, pl, hd.data(), out_w, dx, dy);
      }
  }
  /* HUD digits */
  for (int f = 0; f < 2; f++)
    for (int k = 0; k < TBX_MAX_DIGITS; k++) {
      const int d = tbx_digit_at(fields[f], k);
      if (d < 0) continue;
      const TbxDigitPatch &P = patches[(f * 10 + k) * 10 + d];
      for (int r = 0; r < P.h; r++) for (int cc = 0; cc < P.w; cc++) out[(P.y0 + r) * out_w + P.x0 + cc] = P.px[r * P.w + cc];
    }
  /* movers */
  for (int m = 0; m < BRK_N_MOVERS; m++) {
    if (mv[m].x0 >= mv[m].x1) continue;
    const int sx0 = pl.xs0[fx0[m]], sx1 = pl.xs0[fx1[m]] + TBX_AREA_MAX_TAPS, sy0 = pl.ys0[fy0[m]], sy1 = pl.ys0[fy1[m]] + TBX_AREA_MAX_TAPS;
    uint32_t near = 0;
    for (int q = 0; q < BRK_N_MOVERS; q++)
      if (mv[q].x0 < mv[q].x1 && mv[q].x0 < sx1 && mv[q].x1 > sx0 && mv[q].y0 < sy1 && mv[q].y1 > sy0) near |= 1u << q;
    const bool wall = sy0 < A.wy0 + A.nrows * A.bh && sy1 > A.wy0;
    for (int dy = fy0[m]; dy <= fy1[m]; dy++)
      for (int dx = fx0[m]; dx <= fx1[m]; dx++)
        out[dy * out_w + dx] = brk_direct_pixel<TBX_AREA_MAX_TAPS, TBX_AREA_MAX_TAPS>(A, pl, base0.data(), alive, mv, near, wall, dx, dy);
  }
  return 0;
}

/* Space Invaders' score strip (TbxSiDirect.sc_*, si_direct_kernel step 2c) on the host: the full-frame reference with the pixels the
 * score's digits feed overwritten from the digit-pair table, exactly as the kernel indexes it.  Must equal emu_render(mode 3) whenever
 * nothing else reaches into the strip.  Returns 1 when the table does not exist for this size (out = the reference then). */
int emu_si_score_strip(Emu *e, int out_w, int out_h, uint8_t *out) {
  if (e->game != TBX_SPACE_INVADERS) { g_err = "space_invaders only"; return -1; }
  const int W = e->info->width, H = e->info->height;
  if (emu_render(e, 3, out_w, out_h, out) != 0) return -1;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  if (!tbx::build_area_plan(rs, pl)) return 1;
  std::vector<uint32_t> rgba((size_t)W * H);
  std::vector<uint8_t> base0((size_t)W * H);
  tbx::build_base_frame(e->cfg, 0, 0, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base0.data());
  static TbxSiDirect A;
  std::vector<TbxSpritePatch> sp;
  tbx::build_si_direct(e->cfg, rs, pl, base0.data(), A, sp);
  if (!A.ok || !A.sc_ok) return 1;
  const uint32_t *R = e->rec.data();
  int ufx0 = 255, ufx1 = -1, ufy0 = 255, ufy1 = -1, n_sc = 0;
  for (int slot = SI_SLOT_SCORE; slot < SI_SLOT_LIVES; slot++) {
    const TbxPrim p = si_prim(R, slot);
    if (p.h <= 0) continue;
    if (p.bw != 3 || (int)tbx_luma(p.color) != A.sc_gray || p.x < 0 || p.y < 0 || p.x + p.w > W || p.y + p.h > H) return 1;
    const int fx0 = pl.xdlo[p.x], fx1 = pl.xdhi[p.x + p.w - 1], fy0 = pl.ydlo[p.y], fy1 = pl.ydhi[p.y + p.h - 1];
    ufx0 = fx0 < ufx0 ? fx0 : ufx0; ufx1 = fx1 > ufx1 ? fx1 : ufx1; ufy0 = fy0 < ufy0 ? fy0 : ufy0; ufy1 = fy1 > ufy1 ? fy1 : ufy1;
    n_sc++;
  }
  if (!n_sc) return 1;
  const int32_t score = (int32_t)R[TBX_HW(score)];
  for (int dy = ufy0; dy <= ufy1; dy++)
    for (int dx = ufx0; dx <= ufx1; dx++) {
      const int tc = dx - A.sc_dx0, tr = dy - A.sc_dy0;
      if (tc < 0 || tc >= A.sc_ncol || tr < 0 || tr >= A.sc_nrow) continue;
      const int k0 = A.sc_slot[tc];
      if (k0 == 255) continue;
      int da = tbx_digit_at(score, k0), db = k0 + 1 < TBX_MAX_DIGITS ? tbx_digit_at(score, k0 + 1) : -1;
      if (da < 0) da = 10;
      if (db < 0) db = 10;
      out[dy * out_w + dx] = A.sc_px[tc][da][db][tr];
    }
  return 0;
}

/* Which direct INTER_AREA kernel tables the library builds for this config at out_w x out_h (tbx_direct_build runs the same
 * builders): out[0] = ok (0: every env of the size goes to the tile kernel), then Breakout nrows / n_cls, Space Invaders
 * n_sets (0: no sprite patch tables) / sc_ok (0: no score strip), unused entries 0; out[3], out[4] = the plan's taps per output
 * column / row (the tile kernel's dual mode takes at most 5 x 4).  Returns -1 for a size the library refuses. */
int emu_direct_info(Emu *e, int out_w, int out_h, int32_t *out) {
  const int W = e->info->width, H = e->info->height;
  tbx::ResizeTab rs;
  TbxAreaPlan pl;
  try { tbx::build_resize(W, H, out_w, out_h, rs); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  if (!tbx::build_area_plan(rs, pl)) { g_err = "size pair outside the fused kernel's limits"; return -1; }
  const BrkTable *dt = e->game == TBX_BREAKOUT ? &e->brk_tables[e->cfg.brk.default_tbl] : 0;
  std::vector<uint32_t> rgba((size_t)W * H);
  std::vector<uint8_t> base0((size_t)W * H);
  tbx::build_base_frame(e->cfg, dt, 0, rgba.data());
  tbx::frame_to_gray(rgba.data(), W * H, base0.data());
  out[0] = out[1] = out[2] = 0;
  out[3] = pl.tx; out[4] = pl.ty;
  if (e->game == TBX_BREAKOUT) {
    std::unique_ptr<TbxBrkDirect> A(new TbxBrkDirect);
    tbx::build_brk_direct(e->cfg, *dt, rs, pl, base0.data(), *A);
    out[0] = A->ok; out[1] = A->nrows; out[2] = A->n_cls;
  } else if (e->game == TBX_AMIDAR) {
    std::unique_ptr<TbxAmiDirect> A(new TbxAmiDirect);
    tbx::build_ami_direct(e->cfg, rs, pl, *A);
    out[0] = A->ok;
  } else {
    std::unique_ptr<TbxSiDirect> A(new TbxSiDirect);
    std::vector<TbxSpritePatch> patches;
    tbx::build_si_direct(e->cfg, rs, pl, base0.data(), *A, patches);
    out[0] = A->ok; out[1] = A->n_sets; out[2] = A->sc_ok;
  }
  return 0;
}

char *emu_state_to_json(Emu *e) {
  try {
    Value v;
    if (e->game == TBX_BREAKOUT) { const BrkRec &r = *reinterpret_cast<const BrkRec *>(e->rec.data()); v = tbx::brk_state_to_json(r, e->brk_tables[r.hdr.tbl]); }
    else if (e->game == TBX_AMIDAR) { const AmiRec &r = *reinterpret_cast<const AmiRec *>(e->rec.data()); v = tbx::ami_state_to_json(r, e->ami_tables[r.hdr.tbl]); }
    else v = tbx::si_state_to_json(*reinterpret_cast<const SiRec *>(e->rec.data()));
    return dup_str(tbxjson::dump(v));
  } catch (const std::exception &ex) { g_err = ex.what(); return 0; }
}
int emu_state_from_json(Emu *e, const char *json) {
  std::vector<uint32_t> rec = e->rec;
  try {
    Value v = tbxjson::parse(json);
    if (e->game == TBX_BREAKOUT) { BrkTable t; BrkRec &r = *reinterpret_cast<BrkRec *>(rec.data()); tbx::brk_state_from_json(v, r, t); tbx::brk_mark_delta_ok(e->cfg, t); r.hdr.tbl = intern(e->brk_tables, t); }
    else if (e->game == TBX_AMIDAR) { AmiTable t; AmiRec &r = *reinterpret_cast<AmiRec *>(rec.data()); tbx::ami_state_from_json(v, r, t); r.hdr.tbl = intern(e->ami_tables, t); }
    else tbx::si_state_from_json(v, *reinterpret_cast<SiRec *>(rec.data()));
  } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  e->rec = rec;
  return 0;
}
char *emu_config_to_json(Emu *e) { return dup_str(tbxjson::dump(tbx::config_to_json(e->cfg))); }
int emu_config_from_json(Emu *e, const char *json) {
  tbx::Config c = e->cfg;
  try { tbx::config_from_json(c, tbxjson::parse(json)); } catch (const std::exception &ex) { g_err = ex.what(); return -1; }
  e->cfg = c;
  install_default_table(e);
  return 0;
}
char *emu_query_json(Emu *e, const char *query, const char *args_json) {
  try {
    const BrkTable *brk = e->game == TBX_BREAKOUT ? &e->brk_tables[reinterpret_cast<const BrkRec *>(e->rec.data())->hdr.tbl] : 0;
    return dup_str(tbxjson::dump(tbx::query_json(e->game, e->rec.data(), brk, query, tbxjson::parse(args_json ? args_json : "null"))));
  } catch (const std::exception &ex) { g_err = ex.what(); return 0; }
}
char *emu_schema_for_state(const char *game) { return dup_str(tbxjson::dump(tbx::schema_for_state(tbx::game_from_name(game)))); }
char *emu_schema_for_config(const char *game) { return dup_str(tbxjson::dump(tbx::schema_for_config(tbx::game_from_name(game)))); }
int emu_n_tables(Emu *e) { return (int)(e->game == TBX_BREAKOUT ? e->brk_tables.size() : e->ami_tables.size()); }
uint32_t emu_action_index(uint64_t seed, uint64_t env, uint64_t t, uint32_t n_legal) { return tbx_action_index(seed, env, t, n_legal); }
int emu_ale_action_to_input(int a) { return tbx_ale_action_to_input(a); }

} /* extern "C" */
