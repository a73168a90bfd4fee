/* tbx_host.cpp -- see tbx_host.h.  Pure host C++ (no CUDA): built into libtoybox_b200.so and, for the
 * CPU-only test tier, into tests/emu/libtbx_emu.so. */
#include "tbx_host.h"
#include "tbx_breakout.h"
#include "tbx_space_invaders.h"
#include "tbx_amidar.h"
#include "tbx_direct.h"
#include <errno.h>
#include <math.h>
#include <string.h>

using tbxjson::Value;

namespace tbx {

static void fail(const std::string &m) { throw std::runtime_error(m); }

static const GameInfo GAMES[3] = {
    {TBX_BREAKOUT, "breakout", TBX_BRK_W, TBX_BRK_H, 4, {0, 1, 3, 4}, TBX_WORDS(BrkRec), BRK_N_SLOTS, 2},
    {TBX_AMIDAR, "amidar", TBX_AMI_W, TBX_AMI_H, 10, {0, 1, 2, 3, 4, 5, 10, 11, 12, 13}, TBX_WORDS(AmiRec), AMI_N_SLOTS, 1},
    {TBX_SPACE_INVADERS, "space_invaders", TBX_SI_W, TBX_SI_H, 6, {0, 1, 3, 4, 11, 12}, TBX_WORDS(SiRec), SI_N_SLOTS, 2},
};
const GameInfo *game_info(int game) { return game >= 0 && game < 3 ? &GAMES[game] : 0; }
int game_from_name(const char *name) {
  if (!name) return -1;
  for (int g = 0; g < 3; g++) if (strcmp(GAMES[g].name, name) == 0) return g;
  if (strcmp(name, "spaceinvaders") == 0) return TBX_SPACE_INVADERS;
  return -1;
}

/* ------------------------------------------------------------------ small JSON helpers */
static Value jcolor(uint32_t c) {
  Value v = Value::object();
  v.set("r", Value::integer(c & 255)).set("g", Value::integer((c >> 8) & 255)).set("b", Value::integer((c >> 16) & 255)).set("a", Value::integer(c >> 24));
  return v;
}
static uint32_t ucolor(const Value &v) {
  uint32_t out = 0;
  const char *k[4] = {"r", "g", "b", "a"};
  for (int n = 0; n < 4; n++) {
    int64_t x = v.at(k[n]).as_i64();
    if (x < 0) x = 0;
    if (x > 255) x = 255;
    out |= (uint32_t)x << (8 * n);
  }
  return out;
}
static Value jvec(double x, double y) { Value v = Value::object(); v.set("x", Value::number(x)).set("y", Value::number(y)); return v; }
static Value jrand(const uint64_t s[2]) {
  Value st = Value::array();
  st.push(Value::uinteger(s[0])).push(Value::uinteger(s[1]));
  Value v = Value::object();
  v.set("state", st);
  return v;
}
static void urand(const Value &v, uint64_t s[2]) {
  const Value &st = v.at("state");
  if (st.size() != 2) fail("rand.state must hold two integers");
  s[0] = st.at((size_t)0).as_u64();
  s[1] = st.at((size_t)1).as_u64();
}
static const char *DIRS[4] = {"Up", "Down", "Left", "Right"};
static int udir(const Value &v) {
  const std::string &s = v.as_str();
  for (int d = 0; d < 4; d++) if (s == DIRS[d]) return d;
  fail("unknown direction '" + s + "'");
  return 0;
}
static Value jopt(int32_t v) { return v == TBX_NONE ? Value() : Value::integer(v); }
static int32_t uopt(const Value &v) { return v.is_null() ? TBX_NONE : v.as_i32(); }

/* ------------------------------------------------------------------ default configs */
static const double DEG2RAD = 0.017453292519943295;

void brk_finish_cfg(BrkCfg &c) {
  if (c.n_rows < 0 || c.n_rows > TBX_BRK_MAX_ROWS) fail("breakout: row_scores/row_colors support at most 8 rows");
  if (c.n_starts < 1 || c.n_starts > TBX_BRK_MAX_STARTS) fail("breakout: 1..8 ball_start_positions supported");
  if (c.paddle_discrete_segments < 1 || c.paddle_discrete_segments > TBX_BRK_MAX_SEGS) fail("breakout: paddle_discrete_segments must be 1..16");
  for (int i = 0; i < c.n_starts; i++) {
    volatile double rad = c.start_angle[i] * DEG2RAD;
    c.start_cos[i] = cos(rad);
    c.start_sin[i] = sin(rad);
  }
  int nseg = c.paddle_discrete_segments;
  for (int seg = 0; seg < TBX_BRK_MAX_SEGS; seg++) {
    int s = seg < nseg ? seg : nseg - 1;
    volatile double ang = nseg > 1 ? 150.0 - (double)s * (120.0 / (double)(nseg - 1)) : 90.0;
    volatile double rad = ang * DEG2RAD;
    c.seg_cos[seg] = cos(rad);
    c.seg_sin[seg] = sin(rad);
  }
}

static uint32_t board_char(char ch) { return ch == '=' ? TBX_TILE_UNPAINTED : ch == 'p' ? TBX_TILE_PAINTED : ch == 'c' ? TBX_TILE_CHASE : TBX_TILE_EMPTY; }
static void set_board_row(AmiCfg &c, int ty, const char *row) {
  c.board[ty][0] = c.board[ty][1] = 0;
  for (int tx = 0; tx < TBX_AMI_BW; tx++) c.board[ty][tx >> 4] |= board_char(row[tx]) << (2 * (tx & 15));
}
static const char *AMI_DEFAULT_BOARD[TBX_AMI_BH] = {
    "c========================c======", "=     =   =   =  =   =   =     =", "=     =   =   =  =   =   =     =",
    "=     =   =   =  =   =   =     =", "=     =   =   =  =   =   =     =", "=     =   =   =  =   =   =     =",
    "================================", "=   =    =  =      =  =    =   =", "=   =    =  =      =  =    =   =",
    "=   =    =  =      =  =    =   =", "=   =    =  =      =  =    =   =", "=   =    =  =      =  =    =   =",
    "================================", "=  =       =        =       =  p", "=  =       =        =       =  p",
    "=  =       =        =       =  p", "=  =       =        =       =  p", "=  =       =        =       =  p",
    "===============================p", "=    =        =  =        =    =", "=    =        =  =        =    =",
    "=    =        =  =        =    =", "=    =        =  =        =    =", "=    =        =  =        =    =",
    "c========================c======", "=     =     =      =     =     =", "=     =     =      =     =     =",
    "=     =     =      =     =     =", "=     =     =      =     =     =", "=     =     =      =     =     =",
    "================================"};
/* enemy patrol loops (tile ids ty*32+tx); the reference's tables are compiled into ctoybox and not in
 * the repository, these honour the fixture's enemy start tiles 0, 0, 7, 800, 969 */
static const int32_t AMI_DEFAULT_ROUTES[5][5] = {
    {0, 31, 223, 192, -1}, {0, 384, 415, 31, -1}, {7, 31, 415, 384, 0}, {800, 960, 991, 799, 768}, {969, 991, 607, 576, 960}};

void default_config(int game, Config &cfg) {
  memset(&cfg, 0, sizeof cfg);
  cfg.game = game;
  TbxRng g;
  if (game == TBX_BREAKOUT) {
    BrkCfg &c = cfg.brk;
    static const uint32_t rows[6][3] = {{200, 72, 72}, {198, 108, 58}, {180, 122, 48}, {162, 162, 42}, {72, 160, 72}, {66, 72, 200}};
    static const int32_t scores[6] = {7, 7, 4, 4, 1, 1};
    static const double starts[4][3] = {{24, 80, 30}, {120, 80, 30}, {120, 80, 150}, {216, 80, 150}};
    c.bg_color = tbx_rgba(0, 0, 0, 255);
    c.frame_color = tbx_rgba(144, 144, 144, 255);
    c.paddle_color = c.ball_color = tbx_rgba(200, 72, 72, 255);
    c.n_rows = 6;
    for (int i = 0; i < 6; i++) { c.row_colors[i] = tbx_rgba(rows[i][0], rows[i][1], rows[i][2], 255); c.row_scores[i] = scores[i]; }
    c.start_lives = 5; c.paddle_discrete_segments = 5; c.ball_speed_row_depth = 3;
    c.ball_speed_slow = 2.0; c.ball_speed_fast = 4.0;
    c.n_starts = 4;
    for (int i = 0; i < 4; i++) { c.start_x[i] = starts[i][0]; c.start_y[i] = starts[i][1]; c.start_angle[i] = starts[i][2]; }
    tbx_rng_seed(g, 13);
    c.rand[0] = g.s0; c.rand[1] = g.s1;
    brk_finish_cfg(c);
  } else if (game == TBX_SPACE_INVADERS) {
    SiCfg &c = cfg.si;
    static const int32_t rs[6] = {30, 30, 20, 20, 10, 10};
    c.jitter = 0.5; c.enemy_protocol = 0; c.start_lives = 3;
    c.shields[0][0] = 84; c.shields[1][0] = 148; c.shields[2][0] = 212;
    for (int i = 0; i < 3; i++) c.shields[i][1] = 157;
    for (int i = 0; i < 6; i++) c.row_scores[i] = rs[i];
    tbx_rng_seed(g, 17);
    c.rand[0] = g.s0; c.rand[1] = g.s1;
  } else if (game == TBX_AMIDAR) {
    AmiCfg &c = cfg.ami;
    c.bg_color = tbx_rgba(0, 0, 0, 255);
    c.player_color = tbx_rgba(255, 255, 153, 255);
    c.unpainted_color = tbx_rgba(148, 0, 211, 255);
    c.painted_color = tbx_rgba(255, 255, 30, 255);
    c.enemy_color = tbx_rgba(255, 50, 100, 255);
    c.inner_painted_color = tbx_rgba(255, 255, 0, 255);
    c.start_lives = 3; c.start_jumps = 4; c.chase_time = 300; c.chase_score_bonus = 100;
    c.jump_time = 75; c.box_bonus = 50; c.render_images = 1; c.default_board_bugs = 1;
    c.player_start_tx = 31; c.player_start_ty = 15;
    for (int ty = 0; ty < TBX_AMI_BH; ty++) set_board_row(c, ty, AMI_DEFAULT_BOARD[ty]);
    c.n_enemies = 5;
    for (int i = 0; i < 5; i++) { c.enemies[i].kind = TBX_AI_LOOKUP; c.enemies[i].next = 0; c.enemies[i].default_route_index = i; }
    c.n_routes = 5;
    for (int i = 0; i < 5; i++) {
      int n = 0;
      while (n < 5 && AMI_DEFAULT_ROUTES[i][n] >= 0) { c.routes[i][n] = AMI_DEFAULT_ROUTES[i][n]; n++; }
      c.route_len[i] = n;
    }
    tbx_rng_seed(g, 13);
    c.rand[0] = g.s0; c.rand[1] = g.s1;
  } else fail("unknown game id");
}

/* ------------------------------------------------------------------ geometry tables */
void brk_finish_table(BrkTable &t) {
  int n = t.n_bricks;
  for (int k = 0; k < 5; k++) { int m = n - 32 * k; t.all_mask[k] = m >= 32 ? 0xffffffffu : m <= 0 ? 0u : ((1u << m) - 1u); t.destructible[k] &= t.all_mask[k]; }
  t.bb_x0 = t.bb_y0 = INFINITY; t.bb_x1 = t.bb_y1 = -INFINITY;
  for (int i = 0; i < TBX_BRK_MAX_BRICKS; i++) {
    if (i >= n) { t.px[i] = t.py[i] = t.sx[i] = t.sy[i] = 0; t.points[i] = t.depth[i] = t.row[i] = t.col[i] = 0; t.color[i] = 0; }
    volatile double x1 = t.px[i] + t.sx[i], y1 = t.py[i] + t.sy[i];
    t.x1[i] = x1; t.y1[i] = y1;
    t.ix[i] = tbx_d2i(t.px[i]); t.iy[i] = tbx_d2i(t.py[i]); t.iw[i] = tbx_d2i(t.sx[i]); t.ih[i] = tbx_d2i(t.sy[i]);
    if (i < n) {
      if (t.px[i] < t.bb_x0) t.bb_x0 = t.px[i];
      if (t.py[i] < t.bb_y0) t.bb_y0 = t.py[i];
      if (t.x1[i] > t.bb_x1) t.bb_x1 = t.x1[i];
      if (t.y1[i] > t.bb_y1) t.bb_y1 = t.y1[i];
    }
  }
  if (n == 0) { t.bb_x0 = t.bb_y0 = t.bb_x1 = t.bb_y1 = 0; }
  /* NaN coordinates never compare true in the step; make the early-out box permissive in that case */
  if (!(t.bb_x0 == t.bb_x0) || !(t.bb_y0 == t.bb_y0) || !(t.bb_x1 == t.bb_x1) || !(t.bb_y1 == t.bb_y1)) { t.bb_x0 = t.bb_y0 = -INFINITY; t.bb_x1 = t.bb_y1 = INFINITY; }
  for (int i = 0; i < n; i++) if (t.px[i] != t.px[i] || t.py[i] != t.py[i] || t.x1[i] != t.x1[i] || t.y1[i] != t.y1[i]) { t.bb_x0 = t.bb_y0 = -INFINITY; t.bb_x1 = t.bb_y1 = INFINITY; }
  /* regular column-major grid?  (the default table always is; a table edited through JSON usually is not) */
  t.grid = 0; t.g_ncols = t.g_nrows = 0; t._padg = 0; t.gx0 = t.gy0 = t.ginv_w = t.ginv_h = 0.0;
  if (n > 0 && t.sx[0] > 0.0 && t.sy[0] > 0.0) {
    int nrows = 1;
    while (nrows < n && t.px[nrows] == t.px[0]) nrows++;
    if (n % nrows == 0) {
      const int ncols = n / nrows;
      bool ok = true;
      for (int i = 0; i < n && ok; i++) {
        const int col = i / nrows, row = i % nrows;
        ok = t.px[i] == t.px[0] + col * t.sx[0] && t.py[i] == t.py[0] + row * t.sy[0] && t.sx[i] == t.sx[0] && t.sy[i] == t.sy[0];
      }
      if (ok) { t.grid = 1; t.g_ncols = ncols; t.g_nrows = nrows; t.gx0 = t.px[0]; t.gy0 = t.py[0]; t.ginv_w = 1.0 / t.sx[0]; t.ginv_h = 1.0 / t.sy[0]; }
    }
  }
  t.hud_clear = 1;
  for (int i = 0; i < n; i++) if (t.iw[i] > 0 && t.ih[i] > 0 && t.iy[i] < 12) t.hud_clear = 0;
  t.disjoint = 1;
  for (int i = 0; i < n && t.disjoint; i++)
    for (int j = i + 1; j < n; j++) {
      bool sep = t.ix[i] + t.iw[i] <= t.ix[j] || t.ix[j] + t.iw[j] <= t.ix[i] || t.iy[i] + t.ih[i] <= t.iy[j] || t.iy[j] + t.ih[j] <= t.iy[i];
      if (!sep && t.iw[i] > 0 && t.ih[i] > 0 && t.iw[j] > 0 && t.ih[j] > 0) { t.disjoint = 0; break; }
    }
}
void brk_default_table(const BrkCfg &c, BrkTable &t) {
  memset(&t, 0, sizeof t);
  t.n_bricks = 18 * c.n_rows;
  for (int col = 0; col < 18; col++)
    for (int row = 0; row < c.n_rows; row++) { /* column-major: bricks[i].col = i / n_rows */
      int i = col * c.n_rows + row;
      t.px[i] = 12.0 + 12.0 * col; t.py[i] = 43.0 + 4.0 * row; t.sx[i] = 12.0; t.sy[i] = 4.0;
      t.color[i] = c.row_colors[row]; t.points[i] = c.row_scores[row]; t.depth[i] = c.n_rows - 1 - row;
      t.row[i] = row; t.col[i] = col;
      t.destructible[i >> 5] |= 1u << (i & 31);
    }
  brk_finish_table(t);
}

static int cfg_tile(const AmiCfg &c, int tx, int ty) {
  if (tx < 0 || tx >= TBX_AMI_BW || ty < 0 || ty >= TBX_AMI_BH) return TBX_TILE_EMPTY;
  return (int)((c.board[ty][tx >> 4] >> (2 * (tx & 15))) & 3u);
}
void ami_finish_table(AmiTable &t) {
  t.all_boxes = t.n_boxes >= 32 ? 0xffffffffu : ((1u << t.n_boxes) - 1u);
  t.triggers_chase &= t.all_boxes;
  memset(t.junction_bits, 0, sizeof t.junction_bits);
  for (int i = 0; i < t.n_junctions; i++) {
    int id = t.junctions[i];
    if (id >= 0 && id < TBX_AMI_BW * TBX_AMI_BH) t.junction_bits[id >> 5] |= 1u << (id & 31);
  }
  for (int i = 0; i < t.n_boxes; i++)
    if (t.tl_tx[i] < 0 || t.tl_ty[i] < 0 || t.br_tx[i] >= TBX_AMI_BW || t.br_ty[i] >= TBX_AMI_BH || t.tl_tx[i] > t.br_tx[i] || t.tl_ty[i] > t.br_ty[i])
      fail("amidar: box corners must lie on the 32x31 board with top_left <= bottom_right");
}
void ami_default_table(const AmiCfg &c, AmiTable &t) {
  memset(&t, 0, sizeof t);
  for (int ty = 0; ty < TBX_AMI_BH; ty++)
    for (int tx = 0; tx < TBX_AMI_BW; tx++) {
      bool w = cfg_tile(c, tx, ty) != 0;
      bool h = cfg_tile(c, tx - 1, ty) != 0 || cfg_tile(c, tx + 1, ty) != 0;
      bool v = cfg_tile(c, tx, ty - 1) != 0 || cfg_tile(c, tx, ty + 1) != 0;
      if (w && h && v && t.n_junctions < TBX_AMI_MAX_JUNCTIONS) t.junctions[t.n_junctions++] = ty * TBX_AMI_BW + tx;
      if (cfg_tile(c, tx, ty) == TBX_TILE_CHASE && t.n_chase_junctions < 4) t.chase_junctions[t.n_chase_junctions++] = ty * TBX_AMI_BW + tx;
    }
  /* boxes: maximal empty rectangles; a box's top-left is a walkable tile whose right and lower
   * neighbours are walkable and whose diagonal is empty */
  for (int ty = 0; ty + 1 < TBX_AMI_BH; ty++)
    for (int tx = 0; tx + 1 < TBX_AMI_BW; tx++) {
      if (!(cfg_tile(c, tx, ty) && cfg_tile(c, tx + 1, ty) && cfg_tile(c, tx, ty + 1) && !cfg_tile(c, tx + 1, ty + 1))) continue;
      int bx = tx + 1, by = ty + 1;
      while (bx < TBX_AMI_BW && !cfg_tile(c, bx, ty + 1)) bx++;
      while (by < TBX_AMI_BH && !cfg_tile(c, tx + 1, by)) by++;
      if (bx >= TBX_AMI_BW || by >= TBX_AMI_BH || t.n_boxes >= TBX_AMI_MAX_BOXES) continue;
      int i = t.n_boxes++;
      t.tl_tx[i] = tx; t.tl_ty[i] = ty; t.br_tx[i] = bx; t.br_ty[i] = by;
      if (cfg_tile(c, tx, ty) == TBX_TILE_CHASE) t.triggers_chase |= 1u << i;
    }
  ami_finish_table(t);
}

/* ------------------------------------------------------------------ config JSON */
static const char *SI_PROTOCOLS[2] = {"TargetPlayer", "Random"};
static const char *AI_NAMES[6] = {"Player", "EnemyLookupAI", "EnemyPerimeterAI", "EnemyAmidarMvmt", "EnemyTargetPlayer", "EnemyRandomMvmt"};

static Value jtile(int tx, int ty) { Value v = Value::object(); v.set("tx", Value::integer(tx)).set("ty", Value::integer(ty)); return v; }
static Value jai(const AmiAi &a) {
  if (a.kind == TBX_AI_PLAYER) return Value::string("Player");
  Value kw = Value::object();
  Value st = jtile(a.start_tx, a.start_ty);
  switch (a.kind) {
    case TBX_AI_LOOKUP: kw.set("next", Value::integer(a.next)).set("default_route_index", Value::integer(a.default_route_index)); break;
    case TBX_AI_PERIMETER: kw.set("start", st); break;
    case TBX_AI_AMIDAR:
      kw.set("vert", Value::string(DIRS[a.vert & 3])).set("horiz", Value::string(DIRS[a.horiz & 3]));
      kw.set("start_vert", Value::string(DIRS[a.start_vert & 3])).set("start_horiz", Value::string(DIRS[a.start_horiz & 3])).set("start", st);
      break;
    case TBX_AI_TARGET:
      kw.set("start", st).set("start_dir", Value::string(DIRS[a.start_dir & 3])).set("vision_distance", Value::integer(a.vision_distance));
      kw.set("dir", Value::string(DIRS[a.dir & 3])).set("player_seen", a.has_seen ? jtile(a.seen_tx, a.seen_ty) : Value());
      break;
    default: kw.set("start", st).set("start_dir", Value::string(DIRS[a.start_dir & 3])).set("dir", Value::string(DIRS[a.dir & 3])); break;
  }
  Value v = Value::object();
  v.set(AI_NAMES[a.kind >= 1 && a.kind <= 5 ? a.kind : 5], kw);
  return v;
}
static void uai(const Value &v, AmiAi &a) {
  memset(&a, 0, sizeof a);
  if (v.kind == Value::String) {
    if (v.s != "Player") fail("unknown ai '" + v.s + "'");
    a.kind = TBX_AI_PLAYER;
    return;
  }
  if (v.kind != Value::Object || v.o.size() != 1) fail("ai must be \"Player\" or a single-key object");
  const std::string &name = v.o[0].first;
  const Value &kw = v.o[0].second;
  a.kind = -1;
  for (int k = 1; k <= 5; k++) if (name == AI_NAMES[k]) a.kind = k;
  if (a.kind < 0) fail("unknown ai '" + name + "'");
  if (kw.has("start")) { a.start_tx = kw.at("start").at("tx").as_i32(); a.start_ty = kw.at("start").at("ty").as_i32(); }
  if (kw.has("next")) a.next = kw.at("next").as_i32();
  if (kw.has("default_route_index")) a.default_route_index = kw.at("default_route_index").as_i32();
  if (kw.has("vision_distance")) a.vision_distance = kw.at("vision_distance").as_i32();
  if (kw.has("vert")) a.vert = udir(kw.at("vert"));
  if (kw.has("horiz")) a.horiz = udir(kw.at("horiz"));
  if (kw.has("start_vert")) a.start_vert = udir(kw.at("start_vert"));
  if (kw.has("start_horiz")) a.start_horiz = udir(kw.at("start_horiz"));
  if (kw.has("start_dir")) a.start_dir = udir(kw.at("start_dir"));
  if (kw.has("dir")) a.dir = udir(kw.at("dir"));
  if (kw.has("player_seen") && !kw.at("player_seen").is_null()) {
    a.has_seen = 1; a.seen_tx = kw.at("player_seen").at("tx").as_i32(); a.seen_ty = kw.at("player_seen").at("ty").as_i32();
  }
}

Value config_to_json(const Config &cfg) {
  Value v = Value::object();
  if (cfg.game == TBX_BREAKOUT) {
    const BrkCfg &c = cfg.brk;
    Value starts = Value::array(), scores = Value::array(), colors = Value::array();
    for (int i = 0; i < c.n_starts; i++) {
      Value p = Value::object();
      p.set("angle_degrees", Value::number(c.start_angle[i])).set("y", Value::number(c.start_y[i])).set("x", Value::number(c.start_x[i]));
      starts.push(p);
    }
    for (int i = 0; i < c.n_rows; i++) { scores.push(Value::integer(c.row_scores[i])); colors.push(jcolor(c.row_colors[i])); }
    v.set("paddle_discrete_segments", Value::integer(c.paddle_discrete_segments)).set("ball_start_positions", starts);
    v.set("start_lives", Value::integer(c.start_lives)).set("row_scores", scores);
    v.set("ball_speed_row_depth", Value::integer(c.ball_speed_row_depth)).set("bg_color", jcolor(c.bg_color)).set("rand", jrand(c.rand));
    v.set("row_colors", colors).set("frame_color", jcolor(c.frame_color)).set("paddle_color", jcolor(c.paddle_color));
    v.set("ball_color", jcolor(c.ball_color)).set("ball_speed_fast", Value::number(c.ball_speed_fast)).set("ball_speed_slow", Value::number(c.ball_speed_slow));
  } else if (cfg.game == TBX_SPACE_INVADERS) {
    const SiCfg &c = cfg.si;
    Value sh = Value::array(), rs = Value::array();
    for (int i = 0; i < 3; i++) { Value p = Value::array(); p.push(Value::integer(c.shields[i][0])).push(Value::integer(c.shields[i][1])); sh.push(p); }
    for (int i = 0; i < 6; i++) rs.push(Value::integer(c.row_scores[i]));
    v.set("jitter", Value::number(c.jitter)).set("shields", sh).set("rand", jrand(c.rand)).set("row_scores", rs);
    v.set("enemy_protocol", Value::string(SI_PROTOCOLS[c.enemy_protocol & 1])).set("start_lives", Value::integer(c.start_lives));
  } else {
    const AmiCfg &c = cfg.ami;
    static const char CH[4] = {' ', '=', 'c', 'p'};
    Value board = Value::array(), enemies = Value::array();
    for (int ty = 0; ty < TBX_AMI_BH; ty++) {
      std::string row;
      for (int tx = 0; tx < TBX_AMI_BW; tx++) row.push_back(CH[cfg_tile(c, tx, ty)]);
      board.push(Value::string(row));
    }
    for (int i = 0; i < c.n_enemies; i++) enemies.push(jai(c.enemies[i]));
    v.set("box_bonus", Value::integer(c.box_bonus)).set("inner_painted_color", jcolor(c.inner_painted_color)).set("jump_time", Value::integer(c.jump_time));
    v.set("render_images", Value::boolean(c.render_images != 0)).set("board", board).set("enemy_color", jcolor(c.enemy_color));
    v.set("chase_time", Value::integer(c.chase_time)).set("rand", jrand(c.rand)).set("painted_color", jcolor(c.painted_color));
    v.set("enemies", enemies).set("start_lives", Value::integer(c.start_lives)).set("player_start", jtile(c.player_start_tx, c.player_start_ty));
    v.set("start_jumps", Value::integer(c.start_jumps)).set("default_board_bugs", Value::boolean(c.default_board_bugs != 0));
    v.set("player_color", jcolor(c.player_color)).set("bg_color", jcolor(c.bg_color)).set("chase_score_bonus", Value::integer(c.chase_score_bonus));
    v.set("unpainted_color", jcolor(c.unpainted_color));
  }
  return v;
}

void config_from_json(Config &cfg, const Value &v) {
  if (v.kind != Value::Object) fail("config must be a JSON object");
  if (cfg.game == TBX_BREAKOUT) {
    BrkCfg c = cfg.brk;
    c.paddle_discrete_segments = v.at("paddle_discrete_segments").as_i32();
    const Value &st = v.at("ball_start_positions");
    if (st.size() < 1 || st.size() > TBX_BRK_MAX_STARTS) fail("breakout: 1..8 ball_start_positions supported");
    c.n_starts = (int)st.size();
    for (int i = 0; i < c.n_starts; i++) { c.start_x[i] = st.at(i).at("x").as_f64(); c.start_y[i] = st.at(i).at("y").as_f64(); c.start_angle[i] = st.at(i).at("angle_degrees").as_f64(); }
    c.start_lives = v.at("start_lives").as_i32();
    const Value &rs = v.at("row_scores"), &rc = v.at("row_colors");
    if (rs.size() > TBX_BRK_MAX_ROWS || rc.size() < rs.size()) fail("breakout: at most 8 rows, one colour per row");
    c.n_rows = (int)rs.size();
    for (int i = 0; i < c.n_rows; i++) { c.row_scores[i] = rs.at(i).as_i32(); c.row_colors[i] = ucolor(rc.at(i)); }
    c.ball_speed_row_depth = v.at("ball_speed_row_depth").as_i32();
    c.bg_color = ucolor(v.at("bg_color")); c.frame_color = ucolor(v.at("frame_color"));
    c.paddle_color = ucolor(v.at("paddle_color")); c.ball_color = ucolor(v.at("ball_color"));
    urand(v.at("rand"), c.rand);
    c.ball_speed_fast = v.at("ball_speed_fast").as_f64(); c.ball_speed_slow = v.at("ball_speed_slow").as_f64();
    brk_finish_cfg(c);
    cfg.brk = c;
  } else if (cfg.game == TBX_SPACE_INVADERS) {
    SiCfg c = cfg.si;
    c.jitter = v.at("jitter").as_f64();
    const std::string &proto = v.at("enemy_protocol").as_str();
    if (proto == SI_PROTOCOLS[0]) c.enemy_protocol = 0; else if (proto == SI_PROTOCOLS[1]) c.enemy_protocol = 1; else fail("unknown enemy_protocol '" + proto + "'");
    c.start_lives = v.at("start_lives").as_i32();
    if (v.at("shields").size() != 3 || v.at("row_scores").size() != 6) fail("space_invaders: exactly 3 shields and 6 row_scores supported");
    for (int i = 0; i < 3; i++) { c.shields[i][0] = v.at("shields").at(i).at((size_t)0).as_i32(); c.shields[i][1] = v.at("shields").at(i).at((size_t)1).as_i32(); }
    for (int i = 0; i < 6; i++) c.row_scores[i] = v.at("row_scores").at(i).as_i32();
    urand(v.at("rand"), c.rand);
    cfg.si = c;
  } else {
    AmiCfg c = cfg.ami;
    c.box_bonus = v.at("box_bonus").as_i32(); c.jump_time = v.at("jump_time").as_i32(); c.chase_time = v.at("chase_time").as_i32();
    c.start_lives = v.at("start_lives").as_i32(); c.start_jumps = v.at("start_jumps").as_i32(); c.chase_score_bonus = v.at("chase_score_bonus").as_i32();
    c.inner_painted_color = ucolor(v.at("inner_painted_color")); c.enemy_color = ucolor(v.at("enemy_color"));
    c.painted_color = ucolor(v.at("painted_color")); c.player_color = ucolor(v.at("player_color"));
    c.bg_color = ucolor(v.at("bg_color")); c.unpainted_color = ucolor(v.at("unpainted_color"));
    c.render_images = v.at("render_images").as_bool(); c.default_board_bugs = v.at("default_board_bugs").as_bool();
    const Value &b = v.at("board");
    if (b.size() != TBX_AMI_BH) fail("amidar: board must have 31 rows");
    for (int ty = 0; ty < TBX_AMI_BH; ty++) {
      const std::string &row = b.at(ty).as_str();
      if (row.size() != TBX_AMI_BW) fail("amidar: board rows must have 32 tiles");
      for (int tx = 0; tx < TBX_AMI_BW; tx++) if (!strchr(" =cp", row[tx])) fail("amidar: unknown board character");
      set_board_row(c, ty, row.c_str());
    }
    const Value &en = v.at("enemies");
    if (en.size() > TBX_AMI_MAX_ENEMIES) fail("amidar: at most 8 enemies supported");
    c.n_enemies = (int)en.size();
    for (int i = 0; i < c.n_enemies; i++) uai(en.at(i), c.enemies[i]);
    c.player_start_tx = v.at("player_start").at("tx").as_i32(); c.player_start_ty = v.at("player_start").at("ty").as_i32();
    if (c.player_start_tx < 0 || c.player_start_tx >= TBX_AMI_BW || c.player_start_ty < 0 || c.player_start_ty >= TBX_AMI_BH) fail("amidar: player_start off the board");
    urand(v.at("rand"), c.rand);
    cfg.ami = c;
  }
}

/* ------------------------------------------------------------------ state JSON: Breakout */
Value brk_state_to_json(const BrkRec &r, const BrkTable &t) {
  Value v = Value::object();
  v.set("score", Value::integer(r.hdr.score)).set("lives", Value::integer(r.hdr.lives)).set("rand", jrand(r.hdr.rand)).set("level", Value::integer(r.hdr.level));
  Value paddle = Value::object();
  paddle.set("velocity", jvec(r.paddle_vx, r.paddle_vy)).set("position", jvec(r.paddle_px, r.paddle_py));
  v.set("paddle", paddle).set("paddle_width", Value::number(r.paddle_width)).set("paddle_speed", Value::number(r.paddle_speed)).set("ball_radius", Value::number(r.ball_radius));
  Value balls = Value::array();
  for (int i = 0; i < r.n_balls && i < TBX_BRK_MAX_BALLS; i++) {
    Value b = Value::object();
    b.set("position", jvec(r.ball[i][0], r.ball[i][1])).set("velocity", jvec(r.ball[i][2], r.ball[i][3]));
    balls.push(b);
  }
  v.set("balls", balls);
  Value bricks = Value::array();
  for (int i = 0; i < t.n_bricks; i++) {
    Value b = Value::object();
    b.set("destructible", Value::boolean((t.destructible[i >> 5] >> (i & 31)) & 1u)).set("depth", Value::integer(t.depth[i])).set("color", jcolor(t.color[i]));
    b.set("alive", Value::boolean((r.alive[i >> 5] >> (i & 31)) & 1u)).set("points", Value::integer(t.points[i])).set("size", jvec(t.sx[i], t.sy[i]));
    b.set("position", jvec(t.px[i], t.py[i])).set("row", Value::integer(t.row[i])).set("col", Value::integer(t.col[i]));
    bricks.push(b);
  }
  v.set("bricks", bricks).set("reset", Value::boolean(r.reset != 0)).set("is_dead", Value::boolean(r.is_dead != 0));
  return v;
}
void brk_state_from_json(const Value &v, BrkRec &r, BrkTable &t) {
  if (v.kind != Value::Object) fail("state must be a JSON object");
  memset(&t, 0, sizeof t);
  r.hdr.score = v.has("score") ? v.at("score").as_i32() : v.at("points").as_i32(); /* fixture era: `points` */
  r.hdr.lives = v.at("lives").as_i32();
  r.hdr.level = v.has("level") ? v.at("level").as_i32() : 1;
  urand(v.at("rand"), r.hdr.rand);
  const Value &p = v.at("paddle");
  r.paddle_vx = p.at("velocity").at("x").as_f64(); r.paddle_vy = p.at("velocity").at("y").as_f64();
  r.paddle_px = p.at("position").at("x").as_f64(); r.paddle_py = p.at("position").at("y").as_f64();
  r.paddle_width = v.at("paddle_width").as_f64(); r.paddle_speed = v.at("paddle_speed").as_f64(); r.ball_radius = v.at("ball_radius").as_f64();
  const Value &balls = v.at("balls"), &bricks = v.at("bricks");
  if (balls.kind != Value::Array || bricks.kind != Value::Array) fail("balls and bricks must be arrays");
  if (balls.size() > TBX_BRK_MAX_BALLS) fail("breakout: at most 4 balls supported");
  if (bricks.size() > TBX_BRK_MAX_BRICKS) fail("breakout: at most 144 bricks supported");
  r.n_balls = (int)balls.size();
  memset(r.ball, 0, sizeof r.ball);
  for (int i = 0; i < r.n_balls; i++) {
    r.ball[i][0] = balls.at(i).at("position").at("x").as_f64(); r.ball[i][1] = balls.at(i).at("position").at("y").as_f64();
    r.ball[i][2] = balls.at(i).at("velocity").at("x").as_f64(); r.ball[i][3] = balls.at(i).at("velocity").at("y").as_f64();
  }
  t.n_bricks = (int)bricks.size();
  memset(r.alive, 0, sizeof r.alive);
  for (int i = 0; i < t.n_bricks; i++) {
    const Value &b = bricks.at(i);
    if (b.at("destructible").as_bool()) t.destructible[i >> 5] |= 1u << (i & 31);
    if (b.at("alive").as_bool()) r.alive[i >> 5] |= 1u << (i & 31);
    t.depth[i] = b.at("depth").as_i32(); t.color[i] = ucolor(b.at("color")); t.points[i] = b.at("points").as_i32();
    t.sx[i] = b.at("size").at("x").as_f64(); t.sy[i] = b.at("size").at("y").as_f64();
    t.px[i] = b.at("position").at("x").as_f64(); t.py[i] = b.at("position").at("y").as_f64();
    t.row[i] = b.at("row").as_i32(); t.col[i] = b.at("col").as_i32();
  }
  r.reset = v.has("reset") ? v.at("reset").as_bool() : 0;
  r.is_dead = v.at("is_dead").as_bool();
  r.hdr.prev_score = r.hdr.score;
  brk_finish_table(t);
}

/* ------------------------------------------------------------------ state JSON: Space Invaders */
static Value jlaser(const SiLaser &l) {
  Value v = Value::object();
  v.set("x", Value::integer(l.x)).set("y", Value::integer(l.y)).set("w", Value::integer(l.w)).set("h", Value::integer(l.h)).set("t", Value::integer(l.t));
  v.set("movement", Value::string(DIRS[l.movement & 3])).set("speed", Value::integer(l.speed)).set("color", jcolor(l.color));
  return v;
}
static void ulaser(const Value &v, SiLaser &l) {
  l.x = v.at("x").as_i32(); l.y = v.at("y").as_i32(); l.w = v.at("w").as_i32(); l.h = v.at("h").as_i32(); l.t = v.at("t").as_i32();
  l.movement = udir(v.at("movement")); l.speed = v.at("speed").as_i32(); l.color = ucolor(v.at("color"));
}
Value si_state_to_json(const SiRec &r) {
  Value v = Value::object();
  v.set("score", Value::integer(r.hdr.score)).set("lives", Value::integer(r.hdr.lives)).set("rand", jrand(r.hdr.rand)).set("level", Value::integer(r.hdr.level));
  Value ship = Value::object();
  ship.set("x", Value::integer(r.ship_x)).set("y", Value::integer(r.ship_y)).set("w", Value::integer(r.ship_w)).set("h", Value::integer(r.ship_h));
  ship.set("speed", Value::integer(r.ship_speed)).set("color", jcolor(r.ship_color)).set("alive", Value::boolean(r.ship_alive != 0));
  ship.set("death_counter", jopt(r.ship_death_counter)).set("death_hit_1", Value::boolean(r.ship_death_hit_1 != 0));
  v.set("ship", ship).set("ship_laser", r.has_ship_laser ? jlaser(r.ship_laser) : Value());
  Value enemies = Value::array();
  for (int i = 0; i < TBX_SI_N_ENEMIES; i++) {
    Value e = Value::object();
    e.set("x", Value::integer(r.en_x[i])).set("y", Value::integer(r.en_y[i])).set("row", Value::integer(r.en_row[i])).set("col", Value::integer(r.en_col[i]));
    e.set("id", Value::integer(r.en_id[i])).set("alive", Value::boolean((r.en_alive[i >> 5] >> (i & 31)) & 1u)).set("points", Value::integer(r.en_points[i]));
    e.set("death_counter", jopt(r.en_death[i]));
    enemies.push(e);
  }
  Value mv = Value::object();
  mv.set("move_counter", Value::integer(r.move_counter)).set("move_dir", Value::string(DIRS[r.move_dir & 3])).set("visual_orientation", Value::boolean(r.visual_orientation != 0));
  v.set("enemies", enemies).set("enemies_movement", mv);
  Value lasers = Value::array();
  for (int i = 0; i < r.n_enemy_lasers && i < TBX_SI_MAX_LASERS; i++) lasers.push(jlaser(r.enemy_lasers[i]));
  v.set("enemy_lasers", lasers);
  Value shields = Value::array();
  Value opaque = jcolor(SI_COLOR_SHIELD), clear = jcolor(0);
  for (int i = 0; i < TBX_SI_N_SHIELDS; i++) {
    Value data = Value::array();
    for (int rr = 0; rr < TBX_SI_SHIELD_H; rr++) {
      Value row = Value::array();
      for (int q = 0; q < TBX_SI_SHIELD_W; q++) row.push(((r.shield_rows[i][rr] >> (15 - q)) & 1u) ? opaque : clear);
      data.push(row);
    }
    Value s = Value::object();
    s.set("x", Value::integer(r.shield_x[i])).set("y", Value::integer(r.shield_y[i])).set("data", data);
    shields.push(s);
  }
  v.set("shields", shields);
  Value ufo = Value::object();
  ufo.set("x", Value::integer(r.ufo_x)).set("y", Value::integer(r.ufo_y)).set("appearance_counter", jopt(r.ufo_appearance_counter)).set("death_counter", jopt(r.ufo_death_counter));
  v.set("ufo", ufo).set("life_display_timer", Value::integer(r.life_display_timer)).set("enemy_shot_delay", Value::integer(r.enemy_shot_delay));
  return v;
}
void si_state_from_json(const Value &v, SiRec &r) {
  if (v.kind != Value::Object) fail("state must be a JSON object");
  r.hdr.score = v.at("score").as_i32(); r.hdr.lives = v.at("lives").as_i32(); urand(v.at("rand"), r.hdr.rand);
  r.hdr.level = v.has("level") ? v.at("level").as_i32() : (v.has("levels_completed") ? v.at("levels_completed").as_i32() : 0) + 1;
  const Value &sh = v.at("ship");
  r.ship_x = sh.at("x").as_i32(); r.ship_y = sh.at("y").as_i32(); r.ship_w = sh.at("w").as_i32(); r.ship_h = sh.at("h").as_i32();
  r.ship_speed = sh.at("speed").as_i32(); r.ship_color = ucolor(sh.at("color")); r.ship_alive = sh.at("alive").as_bool();
  r.ship_death_counter = uopt(sh.at("death_counter")); r.ship_death_hit_1 = sh.at("death_hit_1").as_bool();
  r.has_ship_laser = !v.at("ship_laser").is_null();
  memset(&r.ship_laser, 0, sizeof r.ship_laser);
  if (r.has_ship_laser) ulaser(v.at("ship_laser"), r.ship_laser);
  const Value &en = v.at("enemies"), &ls = v.at("enemy_lasers"), &shd = v.at("shields");
  if (en.size() != TBX_SI_N_ENEMIES) fail("space_invaders: exactly 36 enemies supported");
  if (ls.size() > TBX_SI_MAX_LASERS) fail("space_invaders: at most 4 enemy lasers supported");
  if (shd.size() != TBX_SI_N_SHIELDS) fail("space_invaders: exactly 3 shields supported");
  r.en_alive[0] = r.en_alive[1] = 0;
  for (int i = 0; i < TBX_SI_N_ENEMIES; i++) {
    const Value &e = en.at(i);
    r.en_x[i] = e.at("x").as_i32(); r.en_y[i] = e.at("y").as_i32(); r.en_row[i] = e.at("row").as_i32(); r.en_col[i] = e.at("col").as_i32();
    r.en_id[i] = e.at("id").as_i32(); r.en_points[i] = e.at("points").as_i32(); r.en_death[i] = uopt(e.at("death_counter"));
    if (e.at("alive").as_bool()) r.en_alive[i >> 5] |= 1u << (i & 31);
  }
  if (v.has("enemies_movement")) {
    const Value &m = v.at("enemies_movement");
    r.move_counter = m.at("move_counter").as_i32(); r.move_dir = udir(m.at("move_dir")); r.visual_orientation = m.at("visual_orientation").as_bool();
  } else { /* fixture era: per-enemy fields */
    const Value &e0 = en.at((size_t)0);
    r.move_counter = e0.at("move_counter").as_i32(); r.move_dir = e0.at("move_right").as_bool() ? TBX_DIR_RIGHT : TBX_DIR_LEFT;
    r.visual_orientation = e0.at("orientation_init").as_bool();
  }
  r.n_enemy_lasers = (int)ls.size();
  memset(r.enemy_lasers, 0, sizeof r.enemy_lasers);
  for (int i = 0; i < r.n_enemy_lasers; i++) ulaser(ls.at(i), r.enemy_lasers[i]);
  for (int i = 0; i < TBX_SI_N_SHIELDS; i++) {
    const Value &s = shd.at(i);
    r.shield_x[i] = s.at("x").as_i32(); r.shield_y[i] = s.at("y").as_i32();
    const Value &data = s.at("data");
    if (data.size() != TBX_SI_SHIELD_H) fail("space_invaders: shield sprite must be 18 rows of 16 pixels");
    for (int rr = 0; rr < TBX_SI_SHIELD_H; rr++) {
      if (data.at(rr).size() != TBX_SI_SHIELD_W) fail("space_invaders: shield sprite must be 18 rows of 16 pixels");
      uint32_t bits = 0;
      for (int q = 0; q < TBX_SI_SHIELD_W; q++) if (data.at(rr).at(q).at("a").as_i64() != 0) bits |= 1u << (15 - q);
      r.shield_rows[i][rr] = bits;
    }
  }
  const Value &u = v.at("ufo");
  r.ufo_x = u.at("x").as_i32(); r.ufo_y = u.at("y").as_i32(); r.ufo_appearance_counter = uopt(u.at("appearance_counter")); r.ufo_death_counter = uopt(u.at("death_counter"));
  r.life_display_timer = v.at("life_display_timer").as_i32(); r.enemy_shot_delay = v.at("enemy_shot_delay").as_i32();
  r.hdr.prev_score = r.hdr.score;
  r.hdr.tbl = 0;
}

/* ------------------------------------------------------------------ state JSON: Amidar */
static const char *TILES[4] = {"Empty", "Unpainted", "ChaseMarker", "Painted"};
static Value jmob(const AmiMob &m) {
  Value hist = Value::array();
  for (int i = 0; i < m.n_history && i < TBX_AMI_HIST; i++) hist.push(Value::integer(m.history[i]));
  Value pos = Value::object();
  pos.set("x", Value::integer(m.x)).set("y", Value::integer(m.y));
  Value v = Value::object();
  v.set("history", hist).set("step", m.has_step ? jtile(m.step_tx, m.step_ty) : Value()).set("position", pos);
  v.set("caught", Value::boolean(m.caught != 0)).set("speed", Value::integer(m.speed)).set("ai", jai(m.ai));
  return v;
}
static void umob(const Value &v, AmiMob &m) {
  memset(&m, 0, sizeof m);
  const Value &h = v.at("history");
  if (h.size() > TBX_AMI_HIST) fail("amidar: history longer than 8 is not supported");
  m.n_history = (int)h.size();
  for (int i = 0; i < m.n_history; i++) m.history[i] = h.at(i).as_i32();
  m.has_step = !v.at("step").is_null();
  if (m.has_step) { m.step_tx = v.at("step").at("tx").as_i32(); m.step_ty = v.at("step").at("ty").as_i32(); }
  m.x = v.at("position").at("x").as_i32(); m.y = v.at("position").at("y").as_i32();
  m.caught = v.at("caught").as_bool(); m.speed = v.at("speed").as_i32();
  uai(v.at("ai"), m.ai);
}
Value ami_state_to_json(const AmiRec &r, const AmiTable &t) {
  Value v = Value::object();
  v.set("score", Value::integer(r.hdr.score)).set("lives", Value::integer(r.hdr.lives)).set("rand", jrand(r.hdr.rand)).set("level", Value::integer(r.hdr.level));
  Value enemies = Value::array();
  for (int i = 0; i < r.n_enemies && i < TBX_AMI_MAX_ENEMIES; i++) enemies.push(jmob(r.enemies[i]));
  v.set("enemies", enemies).set("player", jmob(r.player)).set("jumps", Value::integer(r.jumps)).set("jump_timer", Value::integer(r.jump_timer)).set("chase_timer", Value::integer(r.chase_timer));
  Value boxes = Value::array(), tiles = Value::array(), cj = Value::array(), jn = Value::array();
  for (int i = 0; i < t.n_boxes; i++) {
    Value b = Value::object();
    b.set("triggers_chase", Value::boolean((t.triggers_chase >> i) & 1u)).set("top_left", jtile(t.tl_tx[i], t.tl_ty[i]));
    b.set("bottom_right", jtile(t.br_tx[i], t.br_ty[i])).set("painted", Value::boolean((r.box_painted >> i) & 1u));
    boxes.push(b);
  }
  for (int ty = 0; ty < TBX_AMI_BH; ty++) {
    Value row = Value::array();
    for (int tx = 0; tx < TBX_AMI_BW; tx++) row.push(Value::string(TILES[(r.tiles[ty][tx >> 4] >> (2 * (tx & 15))) & 3u]));
    tiles.push(row);
  }
  for (int i = 0; i < t.n_chase_junctions; i++) cj.push(Value::integer(t.chase_junctions[i]));
  for (int i = 0; i < t.n_junctions; i++) jn.push(Value::integer(t.junctions[i]));
  Value board = Value::object();
  board.set("boxes", boxes).set("tiles", tiles).set("height", Value::integer(TBX_AMI_BH)).set("chase_junctions", cj).set("width", Value::integer(TBX_AMI_BW)).set("junctions", jn);
  v.set("board", board);
  return v;
}
void ami_state_from_json(const Value &v, AmiRec &r, AmiTable &t) {
  if (v.kind != Value::Object) fail("state must be a JSON object");
  memset(&t, 0, sizeof t);
  r.hdr.score = v.at("score").as_i32(); r.hdr.lives = v.at("lives").as_i32(); urand(v.at("rand"), r.hdr.rand);
  r.hdr.level = v.has("level") ? v.at("level").as_i32() : 1;
  const Value &en = v.at("enemies");
  if (en.size() > TBX_AMI_MAX_ENEMIES) fail("amidar: at most 8 enemies supported");
  r.n_enemies = (int)en.size();
  memset(r.enemies, 0, sizeof r.enemies);
  for (int i = 0; i < r.n_enemies; i++) umob(en.at(i), r.enemies[i]);
  umob(v.at("player"), r.player);
  r.jumps = v.at("jumps").as_i32(); r.jump_timer = v.at("jump_timer").as_i32(); r.chase_timer = v.at("chase_timer").as_i32();
  const Value &b = v.at("board");
  if (b.at("width").as_i32() != TBX_AMI_BW || b.at("height").as_i32() != TBX_AMI_BH) fail("amidar: only 32x31 boards are supported");
  const Value &boxes = b.at("boxes"), &tiles = b.at("tiles"), &jn = b.at("junctions"), &cj = b.at("chase_junctions");
  if (boxes.size() > TBX_AMI_MAX_BOXES) fail("amidar: at most 32 boxes supported");
  if (jn.size() > TBX_AMI_MAX_JUNCTIONS) fail("amidar: at most 64 junctions supported");
  if (cj.size() > 4) fail("amidar: at most 4 chase junctions supported");
  if (tiles.size() != TBX_AMI_BH) fail("amidar: tiles must have 31 rows");
  t.n_boxes = (int)boxes.size();
  r.box_painted = 0;
  for (int i = 0; i < t.n_boxes; i++) {
    const Value &x = boxes.at(i);
    t.tl_tx[i] = x.at("top_left").at("tx").as_i32(); t.tl_ty[i] = x.at("top_left").at("ty").as_i32();
    t.br_tx[i] = x.at("bottom_right").at("tx").as_i32(); t.br_ty[i] = x.at("bottom_right").at("ty").as_i32();
    if (x.at("painted").as_bool()) r.box_painted |= 1u << i;
    if (x.at("triggers_chase").as_bool()) t.triggers_chase |= 1u << i;
  }
  for (int ty = 0; ty < TBX_AMI_BH; ty++) {
    if (tiles.at(ty).size() != TBX_AMI_BW) fail("amidar: tile rows must have 32 entries");
    r.tiles[ty][0] = r.tiles[ty][1] = 0;
    for (int tx = 0; tx < TBX_AMI_BW; tx++) {
      const std::string &name = tiles.at(ty).at(tx).as_str();
      int k = -1;
      for (int q = 0; q < 4; q++) if (name == TILES[q]) k = q;
      if (k < 0) fail("amidar: unknown tile '" + name + "'");
      r.tiles[ty][tx >> 4] |= (uint32_t)k << (2 * (tx & 15));
    }
  }
  t.n_junctions = (int)jn.size();
  for (int i = 0; i < t.n_junctions; i++) t.junctions[i] = jn.at(i).as_i32();
  t.n_chase_junctions = (int)cj.size();
  for (int i = 0; i < t.n_chase_junctions; i++) t.chase_junctions[i] = cj.at(i).as_i32();
  r.hdr.prev_score = r.hdr.score;
  ami_finish_table(t);
}

/* ------------------------------------------------------------------ queries */
Value query_json(int game, const uint32_t *rec, const BrkTable *brk, const std::string &q, const Value &args) {
  if (game == TBX_AMIDAR && q == "tile_to_world") {
    Value res = Value::array();
    res.push(Value::integer((int64_t)args.at("tx").as_i32() * AMI_TW)).push(Value::integer((int64_t)args.at("ty").as_i32() * AMI_TH));
    return res;
  }
  if (game == TBX_AMIDAR && q == "world_to_tile") {
    Value res = Value::array();
    res.push(Value::integer(ami_floordiv(args.at("x").as_i32(), AMI_TW))).push(Value::integer(ami_floordiv(args.at("y").as_i32(), AMI_TH)));
    return res;
  }
  if (game == TBX_BREAKOUT && brk && (q == "bricks_remaining" || q == "count_channels" || q == "channels")) {
    const BrkRec &r = *reinterpret_cast<const BrkRec *>(rec);
    const BrkTable &t = *brk;
    if (q == "bricks_remaining") {
      int c = 0;
      for (int i = 0; i < t.n_bricks; i++) c += (r.alive[i >> 5] >> (i & 31)) & 1u;
      return Value::integer(c);
    }
    /* a channel is a brick column with no alive brick left */
    Value cols = Value::array();
    int count = 0;
    for (int col = 0; col < 64; col++) {
      bool any = false, open = true;
      for (int i = 0; i < t.n_bricks; i++)
        if (t.col[i] == col) { any = true; if ((r.alive[i >> 5] >> (i & 31)) & 1u) open = false; }
      if (any && open) { count++; cols.push(Value::integer(col)); }
    }
    return q == "count_channels" ? Value::integer(count) : cols;
  }
  fail("unknown query '" + q + "'");
  return Value();
}

/* ------------------------------------------------------------------ JSON schema (draft-07 flavoured, what
 * toybox/interventions/core.py:18-20 and the classes' `expected_keys` read: top-level `required` and
 * per-property `type`/`format`) */
static Value prop(const char *type, const char *format = 0) {
  Value v = Value::object();
  v.set("type", Value::string(type));
  if (format) v.set("format", Value::string(format));
  return v;
}
static Value schema_object(const std::vector<std::pair<const char *, Value> > &props, const char *title) {
  Value p = Value::object(), req = Value::array();
  for (size_t i = 0; i < props.size(); i++) { p.set(props[i].first, props[i].second); req.push(Value::string(props[i].first)); }
  Value v = Value::object();
  v.set("$schema", Value::string("http://json-schema.org/draft-07/schema#")).set("title", Value::string(title)).set("type", Value::string("object"));
  v.set("properties", p).set("required", req);
  return v;
}
typedef std::pair<const char *, Value> P;
Value schema_for_state(int game) {
  std::vector<P> p;
  if (game == TBX_BREAKOUT) {
    p.push_back(P("score", prop("integer", "int32"))); p.push_back(P("lives", prop("integer", "int32"))); p.push_back(P("rand", prop("object")));
    p.push_back(P("level", prop("integer", "int32"))); p.push_back(P("paddle", prop("object"))); p.push_back(P("paddle_width", prop("number", "double")));
    p.push_back(P("paddle_speed", prop("number", "double"))); p.push_back(P("ball_radius", prop("number", "double"))); p.push_back(P("balls", prop("array")));
    p.push_back(P("bricks", prop("array"))); p.push_back(P("reset", prop("boolean"))); p.push_back(P("is_dead", prop("boolean")));
    return schema_object(p, "Breakout");
  }
  if (game == TBX_SPACE_INVADERS) {
    p.push_back(P("score", prop("integer", "int32"))); p.push_back(P("lives", prop("integer", "int32"))); p.push_back(P("rand", prop("object")));
    p.push_back(P("level", prop("integer", "int32"))); p.push_back(P("ship", prop("object"))); p.push_back(P("ship_laser", prop("object")));
    p.push_back(P("enemies", prop("array"))); p.push_back(P("enemies_movement", prop("object"))); p.push_back(P("enemy_lasers", prop("array")));
    p.push_back(P("shields", prop("array"))); p.push_back(P("ufo", prop("object"))); p.push_back(P("life_display_timer", prop("integer", "int32")));
    p.push_back(P("enemy_shot_delay", prop("integer", "int32")));
    return schema_object(p, "SpaceInvaders");
  }
  p.push_back(P("score", prop("integer", "int32"))); p.push_back(P("lives", prop("integer", "int32"))); p.push_back(P("rand", prop("object")));
  p.push_back(P("level", prop("integer", "int32"))); p.push_back(P("enemies", prop("array"))); p.push_back(P("player", prop("object")));
  p.push_back(P("jumps", prop("integer", "int32"))); p.push_back(P("jump_timer", prop("integer", "int32"))); p.push_back(P("chase_timer", prop("integer", "int32")));
  p.push_back(P("board", prop("object")));
  return schema_object(p, "Amidar");
}
Value schema_for_config(int game) {
  Config c;
  default_config(game, c);
  Value js = config_to_json(c);
  std::vector<P> p;
  for (size_t i = 0; i < js.o.size(); i++) {
    const Value &x = js.o[i].second;
    const char *type = x.kind == Value::Bool ? "boolean" : (x.kind == Value::Int || x.kind == Value::UInt) ? "integer" : x.kind == Value::Double ? "number"
                       : x.kind == Value::String ? "string" : x.kind == Value::Array ? "array" : "object";
    p.push_back(P(js.o[i].first.c_str(), prop(type, x.kind == Value::Int ? "int32" : x.kind == Value::Double ? "double" : 0)));
  }
  return schema_object(p, game == TBX_BREAKOUT ? "BreakoutConfig" : game == TBX_AMIDAR ? "AmidarConfig" : "SpaceInvadersConfig");
}

/* ------------------------------------------------------------------ INTER_AREA tap tables
 * OpenCV's general area-resize: destination cell dx covers source [dx*scale, (dx+1)*scale); partial
 * cells at both ends are weighted by the covered fraction, weights normalised by the cell width and
 * rounded to f32.  The kernels accumulate the taps in this table's order. */
static void build_axis(int ssize, int dsize, ResizeAxis &ax) {
  if (dsize < 1 || dsize > TBX_RS_MAX_DST || dsize > ssize) fail("resize: destination must be 1..256 and no larger than the source");
  double scale = 1.0 / ((double)dsize / (double)ssize);
  memset(&ax, 0, sizeof ax);
  ax.ssize = ssize; ax.dsize = dsize;
  int k = 0;
  for (int dx = 0; dx < dsize; dx++) {
    ax.start[dx] = (uint16_t)k;
    double fsx1 = dx * scale, fsx2 = fsx1 + scale;
    double cell = scale < (double)ssize - fsx1 ? scale : (double)ssize - fsx1;
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    if (sx2 > ssize - 1) sx2 = ssize - 1;
    if (sx1 > sx2) sx1 = sx2;
    if (k + (sx2 - sx1) + 2 > TBX_RS_MAX_TAPS) fail("resize: too many taps");
    if (sx1 - fsx1 > 1e-3) { ax.si[k] = (uint16_t)(sx1 - 1); ax.alpha[k++] = (float)((sx1 - fsx1) / cell); }
    for (int sx = sx1; sx < sx2; sx++) { ax.si[k] = (uint16_t)sx; ax.alpha[k++] = (float)(1.0 / cell); }
    if (fsx2 - sx2 > 1e-3) {
      double m = fsx2 - sx2;
      if (m > 1.0) m = 1.0;
      if (m > cell) m = cell;
      ax.si[k] = (uint16_t)sx2; ax.alpha[k++] = (float)(m / cell);
    }
    if (k - ax.start[dx] > ax.max_taps) ax.max_taps = k - ax.start[dx];
    if (k == ax.start[dx]) fail("resize: empty destination cell");
  }
  ax.start[dsize] = (uint16_t)k;
  ax.ntaps = k;
}
void build_resize(int sw, int sh, int dw, int dh, ResizeTab &t) {
  double sx = (double)sw / dw, sy = (double)sh / dh;
  if (dw > sw || dh > sh) fail("resize: only down-sampling is supported (INTER_AREA general path)");
  if (sx == floor(sx) && sy == floor(sy)) fail("resize: integer scale factors take OpenCV's integer fast path, which is not implemented");
  build_axis(sw, dw, t.x);
  build_axis(sh, dh, t.y);
}

bool build_area_plan(const ResizeTab &t, TbxAreaPlan &pl) {
  memset(&pl, 0, sizeof pl);
  const ResizeAxis *ax[2] = {&t.x, &t.y};
  if (t.x.dsize > TBX_AREA_MAX_DST || t.y.dsize > TBX_AREA_MAX_DST || t.x.ssize > TBX_AREA_MAX_SRC || t.y.ssize > TBX_AREA_MAX_SRC) return false;
  if (t.x.max_taps > TBX_AREA_MAX_TAPS || t.y.max_taps > TBX_AREA_MAX_TAPS) return false;
  pl.sw = t.x.ssize; pl.sh = t.y.ssize; pl.dw = t.x.dsize; pl.dh = t.y.dsize; pl.tx = t.x.max_taps; pl.ty = t.y.max_taps;
  for (int a = 0; a < 2; a++) {
    const ResizeAxis &A = *ax[a];
    uint8_t *dlo = a == 0 ? pl.xdlo : pl.ydlo, *dhi = a == 0 ? pl.xdhi : pl.ydhi;
    for (int s = 0; s < TBX_AREA_MAX_SRC; s++) { dlo[s] = 255; dhi[s] = 0; }
    for (int d = 0; d < A.dsize; d++) {
      int k0 = A.start[d], n = A.start[d + 1] - k0;
      for (int k = 0; k < n; k++) if (A.si[k0 + k] != A.si[k0] + k) return false; /* taps must be consecutive */
      (a == 0 ? pl.xs0 : pl.ys0)[d] = A.si[k0];
      if (a == 1) pl.yn[d] = (uint16_t)n;
      for (int k = 0; k < TBX_AREA_MAX_TAPS; k++) (a == 0 ? pl.xalpha : pl.yalpha)[k][d] = k < n ? A.alpha[k0 + k] : 0.0f;
      for (int k = 0; k < n; k++) {
        int si = A.si[k0 + k];
        if (d < dlo[si]) dlo[si] = (uint8_t)d;
        if (d > dhi[si]) dhi[si] = (uint8_t)d;
      }
    }
    /* a source index that feeds nothing (cannot happen when down-sampling) inherits its neighbour's range */
    for (int s = 0; s < A.ssize; s++) if (dlo[s] > dhi[s]) { dlo[s] = s ? dlo[s - 1] : 0; dhi[s] = s ? dhi[s - 1] : 0; }
  }
  return true;
}

int n_static_slots(int game) { return game == TBX_BREAKOUT ? BRK_N_STATIC : game == TBX_AMIDAR ? AMI_N_STATIC : SI_N_STATIC; }
static const uint32_t HOST_BANK[TBX_BANK_WORDS] = TBX_BANK_INIT;
static void paint_prim_host(const TbxPrim &p, const uint32_t *rec, int W, int H, uint32_t *rgba) {
  if (p.h <= 0) return;
  for (int y = p.y < 0 ? 0 : p.y; y < p.y + p.h && y < H; y++)
    for (int x = p.x < 0 ? 0 : p.x; x < p.x + p.w && x < W; x++)
      if (tbx_prim_covers(p, HOST_BANK, rec, x, y)) rgba[(size_t)y * W + x] = p.color;
}
void build_base_frame(const Config &c, const BrkTable *brk_default, int base_id, uint32_t *rgba) {
  const GameInfo *gi = game_info(c.game);
  const int W = gi->width, H = gi->height;
  uint32_t clearv = c.game == TBX_BREAKOUT ? c.brk.bg_color : c.game == TBX_AMIDAR ? c.ami.bg_color : SI_COLOR_BLACK;
  for (int i = 0; i < W * H; i++) rgba[i] = clearv;
  std::vector<uint32_t> rec(gi->rec_words, 0); /* static slots never read the record */
  for (int s = 0; s < n_static_slots(c.game); s++) {
    TbxPrim p = c.game == TBX_BREAKOUT ? brk_prim(rec.data(), c.brk, 0, s) : c.game == TBX_AMIDAR ? ami_prim(rec.data(), c.ami, 0, s) : si_prim(rec.data(), s);
    paint_prim_host(p, rec.data(), W, H, rgba);
  }
  if (base_id != 1) return;
  if (c.game == TBX_BREAKOUT && brk_default) {
    BrkRec &r = *reinterpret_cast<BrkRec *>(rec.data());
    r.hdr.tbl = 0; /* brk_default is passed as table 0 */
    for (int k = 0; k < 5; k++) r.alive[k] = brk_default->all_mask[k];
    for (int s = BRK_SLOT_BRICKS; s < BRK_SLOT_PADDLE; s++) paint_prim_host(brk_prim(rec.data(), c.brk, brk_default, s), rec.data(), W, H, rgba);
  } else if (c.game == TBX_AMIDAR) {
    AmiRec &r = *reinterpret_cast<AmiRec *>(rec.data());
    for (int ty = 0; ty < TBX_AMI_BH; ty++) { r.tiles[ty][0] = c.ami.board[ty][0]; r.tiles[ty][1] = c.ami.board[ty][1]; }
    for (int s = AMI_SLOT_TILES; s < AMI_SLOT_BOXES; s++) paint_prim_host(ami_prim(rec.data(), c.ami, 0, s), rec.data(), W, H, rgba);
  }
}
void brk_mark_delta_ok(const Config &c, BrkTable &t) {
  t.delta_ok = 0;
  if (c.game != TBX_BREAKOUT || !t.disjoint || !t.hud_clear) return;
  std::vector<uint32_t> base0((size_t)TBX_BRK_W * TBX_BRK_H);
  build_base_frame(c, 0, 0, base0.data());
  for (int i = 0; i < t.n_bricks; i++)
    for (int y = t.iy[i] < 0 ? 0 : t.iy[i]; y < t.iy[i] + t.ih[i] && y < TBX_BRK_H; y++)
      for (int x = t.ix[i] < 0 ? 0 : t.ix[i]; x < t.ix[i] + t.iw[i] && x < TBX_BRK_W; x++)
        if (base0[(size_t)y * TBX_BRK_W + x] != c.brk.bg_color) return;
  t.delta_ok = 1;
}
void frame_to_gray(const uint32_t *rgba, int npix, uint8_t *gray) { for (int i = 0; i < npix; i++) gray[i] = (uint8_t)tbx_luma(rgba[i]); }
void area_resize(const uint8_t *gray, const ResizeTab &t, uint8_t *out) {
  const int W = t.x.ssize, H = t.y.ssize, dw = t.x.dsize, dh = t.y.dsize;
  std::vector<float> buf((size_t)H * dw);
  for (int y = 0; y < H; y++) for (int dx = 0; dx < dw; dx++) buf[(size_t)y * dw + dx] = tbx_area_h(gray + (size_t)y * W, t.x, dx);
  for (int dy = 0; dy < dh; dy++) for (int dx = 0; dx < dw; dx++) out[dy * dw + dx] = tbx_area_v(buf.data(), dw, 0, t.y, dy, dx);
}
int digit_slot0(int game) { return game == TBX_BREAKOUT ? BRK_SLOT_SCORE : game == TBX_AMIDAR ? AMI_SLOT_SCORE : SI_SLOT_SCORE; }
int digit_slots(int game) { return game == TBX_BREAKOUT ? BRK_SLOT_BRICKS - BRK_SLOT_SCORE : game == TBX_AMIDAR ? AMI_N_SLOTS - AMI_SLOT_SCORE : SI_SLOT_SHIELDS - SI_SLOT_SCORE; }
/* one output pixel of cv2's INTER_AREA, the arithmetic of area_resize above (tbx_area_h per tap row, accumulated like tbx_area_v) */
static uint8_t area_pixel(const uint8_t *gray, int W, const ResizeTab &t, int dx, int dy) {
  int k = t.y.start[dy], k1 = t.y.start[dy + 1];
  float s = tbx_fmul(t.y.alpha[k], tbx_area_h(gray + (size_t)t.y.si[k] * W, t.x, dx));
  for (k++; k < k1; k++) s = tbx_fadd(s, tbx_fmul(t.y.alpha[k], tbx_area_h(gray + (size_t)t.y.si[k] * W, t.x, dx)));
  int v = tbx_f2i_rn(s);
  return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
}
void build_digit_patches(const Config &c, const BrkTable *brk_default, const ResizeTab &t, const TbxAreaPlan &plan, const uint8_t *base_gray,
                         TbxDigitPatch *out) {
  const GameInfo *gi = game_info(c.game);
  const int W = gi->width, H = gi->height;
  std::vector<uint8_t> gray(base_gray, base_gray + (size_t)W * H);
  std::vector<uint32_t> rec(gi->rec_words, 0);
  memset(out, 0, sizeof(TbxDigitPatch) * TBX_DP_SLOTS * 10);
  const int s0 = digit_slot0(c.game), ns = digit_slots(c.game);
  for (int idx = 0; idx < ns && idx < TBX_DP_SLOTS; idx++) {
    const int k = idx % TBX_MAX_DIGITS; /* decimal position inside its field */
    for (int d = 0; d < 10; d++) {
      /* a field value whose digit at position k is d (and that shows position k at all) */
      long long v = d;
      for (int i = 0; i < k; i++) v *= 10;
      if (d == 0 && k > 0) { v = 1; for (int i = 0; i <= k; i++) v *= 10; }
      if (v > 2000000000LL) continue;
      std::fill(rec.begin(), rec.end(), 0u);
      TbxHdr &h = *reinterpret_cast<TbxHdr *>(rec.data());
      h.score = (int32_t)v; h.lives = (int32_t)v;
      TbxPrim p;
      if (c.game == TBX_BREAKOUT) p = brk_prim(rec.data(), c.brk, brk_default, s0 + idx);
      else if (c.game == TBX_AMIDAR) { reinterpret_cast<AmiRec *>(rec.data())->jumps = (int32_t)v; p = ami_prim(rec.data(), c.ami, 0, s0 + idx); }
      else { reinterpret_cast<SiRec *>(rec.data())->life_display_timer = 1; p = si_prim(rec.data(), s0 + idx); }
      if (p.h <= 0 || p.bw != 3 || p.off != TBX_BANK_FONT + 5 * d) continue; /* not a digit sprite of this value */
      const int x0 = p.x < 0 ? 0 : p.x, x1 = p.x + p.w > W ? W : p.x + p.w, y0 = p.y < 0 ? 0 : p.y, y1 = p.y + p.h > H ? H : p.y + p.h;
      if (x0 >= x1 || y0 >= y1) continue;
      const int dx0 = plan.xdlo[x0], dx1 = plan.xdhi[x1 - 1], dy0 = plan.ydlo[y0], dy1 = plan.ydhi[y1 - 1];
      const int w = dx1 - dx0 + 1, hh = dy1 - dy0 + 1;
      if (w < 1 || hh < 1 || w > 8 || w * hh > TBX_DP_MAX) continue;
      const uint8_t lum = (uint8_t)tbx_luma(p.color);
      for (int y = y0; y < y1; y++)
        for (int x = x0; x < x1; x++)
          if (tbx_prim_covers(p, HOST_BANK, rec.data(), x, y)) gray[(size_t)y * W + x] = lum;
      TbxDigitPatch &P = out[idx * 10 + d];
      P.x0 = (uint8_t)dx0; P.y0 = (uint8_t)dy0; P.w = (uint8_t)w; P.h = (uint8_t)hh;
      for (int r = 0; r < hh; r++)
        for (int cc = 0; cc < w; cc++) P.px[r * w + cc] = area_pixel(gray.data(), W, t, dx0 + cc, dy0 + r);
      for (int y = y0; y < y1; y++) memcpy(&gray[(size_t)y * W + x0], base_gray + (size_t)y * W + x0, (size_t)(x1 - x0));
    }
  }
}

/* ------------------------------------------------------------------ direct INTER_AREA tables (tbx_direct.h) */
/* horizontal sum of one source row at output column dx: the kernels' zero-padded tap order */
static float hsum_row(const uint8_t *row, int W, const TbxAreaPlan &pl, int dx) {
  float h = 0.0f;
  for (int t = 0; t < TBX_AREA_MAX_TAPS; t++) {
    const int x = pl.xs0[dx] + t < W ? pl.xs0[dx] + t : W - 1;
    const float p = tbx_fmul((float)row[x], pl.xalpha[t][dx]);
    h = t == 0 ? p : tbx_fadd(h, p);
  }
  return h;
}
void build_brk_direct(const Config &c, const BrkTable &t, const ResizeTab &rs, const TbxAreaPlan &pl, const uint8_t *base0, TbxBrkDirect &A) {
  memset(&A, 0, sizeof A);
  const int W = TBX_BRK_W, H = TBX_BRK_H, dw = pl.dw, dh = pl.dh;
  if (c.game != TBX_BREAKOUT || !t.delta_ok || dw % 4 != 0 || dw > TBX_AREA_MAX_DST || dh > TBX_AREA_MAX_DST || pl.tx > 5 || pl.ty > 4) return;
  const int n = t.n_bricks, nrows = c.brk.n_rows;
  if (n <= 0 || nrows <= 0 || nrows > TBX_BRK_MAX_ROWS || n % nrows != 0) return;
  const int ncols = n / nrows;
  if (ncols > 31) return;
  const int bw = t.iw[0], bh = t.ih[0], wx0 = t.ix[0], wy0 = t.iy[0];
  if (bw <= 0 || bh <= 0 || wx0 < 0 || wy0 < 0 || wx0 + ncols * bw > W || wy0 + nrows * bh > H) return;
  for (int i = 0; i < n; i++) {
    const int col = i / nrows, row = i % nrows;
    if (t.ix[i] != wx0 + col * bw || t.iy[i] != wy0 + row * bh || t.iw[i] != bw || t.ih[i] != bh) return;
    A.brickgray[i] = (uint8_t)tbx_luma(t.color[i]);
  }
  A.ncols = ncols; A.nrows = nrows; A.wx0 = wx0; A.wy0 = wy0; A.bw = bw; A.bh = bh;
  A.paddle_gray = tbx_luma(c.brk.paddle_color); A.ball_gray = tbx_luma(c.brk.ball_color);
  for (int k = 2; k <= TBX_AREA_MAX_DST; k++) A.inv32[k] = 0xffffffffu / (uint32_t)k + 1u;
  memset(A.xcol, 255, sizeof A.xcol);
  memset(A.yrow, 255, sizeof A.yrow);
  for (int x = wx0; x < wx0 + ncols * bw; x++) A.xcol[x] = (uint8_t)((x - wx0) / bw);
  for (int y = wy0; y < wy0 + nrows * bh; y++) A.yrow[y] = (uint8_t)((y - wy0) / bh);
  /* base frame 0 must look the same on every source row of a brick row (it holds the side walls and background only) */
  for (int r = 0; r < nrows; r++)
    for (int y = wy0 + r * bh + 1; y < wy0 + (r + 1) * bh; y++)
      if (memcmp(base0 + (size_t)y * W, base0 + (size_t)(wy0 + r * bh) * W, W) != 0) return;
  /* per output column: the brick columns its real taps touch -- at most two neighbours -- and the look-up table */
  std::vector<uint8_t> row(W);
  for (int dx = 0; dx < dw; dx++) {
    int cmin = 255, cmax = -1;
    uint32_t cols = 0;
    for (int k = rs.x.start[dx]; k < rs.x.start[dx + 1]; k++) {
      const int cc = A.xcol[rs.x.si[k]];
      if (cc == 255) continue;
      cols |= 1u << cc;
      if (cc < cmin) cmin = cc;
      if (cc > cmax) cmax = cc;
    }
    if (cmax >= 0 && cmax - cmin > 1) return;
    int c0 = cmax < 0 ? 0 : cmin;
    if (c0 > ncols - 2) c0 = ncols - 2 < 0 ? 0 : ncols - 2;
    A.col0[dx] = (uint8_t)c0;
    A.wordcols[dx >> 2] |= cols;
    for (int r = 0; r < nrows; r++)
      for (int bits = 0; bits < 4; bits++) {
        memcpy(row.data(), base0 + (size_t)(wy0 + r * bh) * W, W);
        for (int j = 0; j < 2; j++) {
          const int cc = c0 + j;
          if (cc >= ncols || !((bits >> j) & 1)) continue;
          for (int x = wx0 + cc * bw; x < wx0 + (cc + 1) * bw; x++) row[x] = A.brickgray[cc * nrows + r];
        }
        A.hlut[r][bits][dx] = hsum_row(row.data(), W, pl, dx);
      }
  }
  /* per output row of the wall: which H row every tap reads */
  const int wy1 = wy0 + nrows * bh;
  A.wdy0 = pl.ydlo[wy0]; A.wdy1 = pl.ydhi[wy1 - 1];
  if (A.wdy1 - A.wdy0 + 1 > 32) return;
  for (int dy = A.wdy0; dy <= A.wdy1; dy++) {
    const int nreal = rs.y.start[dy + 1] - rs.y.start[dy];
    for (int k = 0; k < TBX_AREA_MAX_TAPS; k++) {
      if (k >= nreal) { A.hsel[dy][k] = A.hsel[dy][0]; continue; } /* zero weight: any finite row */
      const int y = pl.ys0[dy] + k;
      if (A.yrow[y] != 255) { A.hsel[dy][k] = A.yrow[y]; A.dyrows[dy] |= (uint8_t)(1u << A.yrow[y]); continue; }
      float hrow[TBX_AREA_MAX_DST];
      for (int dx = 0; dx < dw; dx++) hrow[dx] = hsum_row(base0 + (size_t)y * W, W, pl, dx);
      int s = 0;
      for (; s < A.n_static; s++) if (memcmp(A.hstatic[s], hrow, sizeof(float) * dw) == 0) break;
      if (s == A.n_static) {
        if (A.n_static == TBX_BD_MAX_STATIC) return;
        memcpy(A.hstatic[A.n_static++], hrow, sizeof(float) * dw);
      }
      A.hsel[dy][k] = (uint8_t)(nrows + s);
    }
  }
  /* HUD digit rows (score, lives) must stay clear of the wall's output rows */
  {
    std::vector<uint32_t> rec(TBX_WORDS(BrkRec), 0);
    TbxHdr &h = *reinterpret_cast<TbxHdr *>(rec.data());
    h.score = 1999999999; h.lives = 1999999999;
    int y1 = 0;
    for (int s = BRK_SLOT_SCORE; s < BRK_SLOT_BRICKS; s++) { const TbxPrim p = brk_prim(rec.data(), c.brk, &t, s); if (p.h > 0 && p.y + p.h > y1) y1 = p.y + p.h; }
    if (y1 > H) y1 = H;
    A.hud_dyhi = y1 > 0 ? pl.ydhi[y1 - 1] : -1;
    if (A.wdy0 <= A.hud_dyhi) return;
  }
  /* rows of base frame 0 by class */
  A.n_cls = 0;
  for (int y = 0; y < H; y++) {
    int cls = -1;
    for (int k = 0; k < A.n_cls && cls < 0; k++)
      if (memcmp(A.clsrows + (size_t)k * W, base0 + (size_t)y * W, W) == 0) cls = k;
    if (cls < 0) {
      if (A.n_cls == TBX_BD_MAX_CLS) { A.n_cls = 0; break; }
      cls = A.n_cls++;
      memcpy(A.clsrows + (size_t)cls * W, base0 + (size_t)y * W, W);
    }
    A.rowcls[y] = (uint8_t)cls;
  }
  A.ok = 1;
}

void build_brk_img(const TbxBrkDirect &A, const TbxAreaPlan &pl, int tx, int ty, const uint8_t *base1_out, const TbxDigitPatch *patches1, std::vector<uint8_t> &img) {
  const int W = TBX_BRK_W, H = TBX_BRK_H, dw = pl.dw, dh = pl.dh, hs = (dw + 3) & ~3, ps = brk_plan_pitch(dw, dh);
  const TbxBrkImgLayout L = brk_img_layout(tx, ty, dw, dh, A.nrows, A.n_static, A.n_cls);
  img.assign((size_t)L.bytes, 0);
  uint8_t *b = img.data();
  /* the cached digit slots: the first TBX_BRK_DIG_WORDS words of each patch (header, then pixels); the kernel uses them only when
   * every one of them fits */
  int32_t dig_cached = 1;
  for (int e = 0; e < TBX_BRK_DIG_SLOTS * 10; e++) {
    const int cid = e / 10, slot = cid < 4 ? cid : cid + TBX_MAX_DIGITS - 4;
    const TbxDigitPatch &P = patches1[slot * 10 + e % 10];
    if (P.w * P.h > 4 * (TBX_BRK_DIG_WORDS - 1)) dig_cached = 0;
    memcpy(b + TBX_BI_DIG + e * TBX_BRK_DIG_WORDS * 4, &P, TBX_BRK_DIG_WORDS * 4);
  }
  memcpy(b + TBX_BI_FLAGS, &dig_cached, 4);
  memcpy(b + TBX_BI_ROWCLS, A.rowcls, H);
  memcpy(b + TBX_BI_INV, A.inv32, sizeof A.inv32);
  memcpy(b + TBX_BI_XDLO, pl.xdlo, W); memcpy(b + TBX_BI_XDHI, pl.xdhi, W);
  memcpy(b + TBX_BI_YDLO, pl.ydlo, H); memcpy(b + TBX_BI_YDHI, pl.ydhi, H);
  memcpy(b + TBX_BI_XCOL, A.xcol, W); memcpy(b + TBX_BI_YROW, A.yrow, H);
  memcpy(b + TBX_BI_BGRAY, A.brickgray, sizeof A.brickgray);
  memcpy(b + TBX_BI_WORDCOLS, A.wordcols, sizeof A.wordcols);
  memcpy(b + TBX_BI_COL0, A.col0, sizeof A.col0);
  memcpy(b + TBX_BI_DYROWS, A.dyrows, sizeof A.dyrows);
  for (int dy = 0; dy < TBX_AREA_MAX_DST; dy++) memcpy(b + TBX_BI_HSEL + dy * ty, A.hsel[dy], ty);
  memcpy(b + L.base1, base1_out, (size_t)dw * dh);
  /* the plan's weights and first-source indices at pitch ps, entries past the output size repeat its last one */
  float *xa = reinterpret_cast<float *>(b + L.plan), *ya = xa + tx * ps;
  uint16_t *xs = reinterpret_cast<uint16_t *>(ya + ty * ps), *ys = xs + ps;
  for (int i = 0; i < ps; i++) {
    const int jx = i < dw - 1 ? i : dw - 1, jy = i < dh - 1 ? i : dh - 1;
    for (int t = 0; t < tx; t++) xa[t * ps + i] = pl.xalpha[t][jx];
    for (int t = 0; t < ty; t++) ya[t * ps + i] = pl.yalpha[t][jy];
    xs[i] = pl.xs0[jx]; ys[i] = pl.ys0[jy];
  }
  for (int rp = 0; rp < A.nrows * 4; rp++) memcpy(b + L.hlut + (size_t)rp * hs * 4, A.hlut[rp >> 2][rp & 3], sizeof(float) * dw);
  for (int s = 0; s < A.n_static; s++) memcpy(b + L.hstatic + (size_t)s * hs * 4, A.hstatic[s], sizeof(float) * dw);
  memcpy(b + L.cls, A.clsrows, (size_t)A.n_cls * W + 16);
}

/* Space Invaders: the score strip (TbxSiDirect.sc_*): every output pixel the ten digit slots feed, for every pair of digits in the (at
 * most two, neighbouring) slots that feed its column */
static void build_si_score_strip(const ResizeTab &rs, const TbxAreaPlan &pl, const uint8_t *base0, TbxSiDirect &A) {
  const int W = TBX_SI_W, H = TBX_SI_H;
  A.sc_ok = 0;
  A.sc_gray = (int32_t)tbx_luma(SI_COLOR_HUD);
  std::vector<uint32_t> rec(TBX_WORDS(SiRec), 0);
  TbxHdr &hd = *reinterpret_cast<TbxHdr *>(rec.data());
  /* the boxes of the ten slots (a score of ten digits shows them all) */
  int bx0[TBX_MAX_DIGITS], bx1[TBX_MAX_DIGITS], by0 = 0, by1 = 0;
  hd.score = 1999999999;
  for (int k = 0; k < TBX_MAX_DIGITS; k++) {
    const TbxPrim p = si_prim(rec.data(), SI_SLOT_SCORE + k);
    if (p.h <= 0 || p.bw != 3 || p.x < 0 || p.y < 0 || p.x + p.w > W || p.y + p.h > H) return;
    if (k > 0 && (p.y != by0 || p.y + p.h != by1 || p.x + p.w > bx0[k - 1])) return; /* one row of boxes, right to left */
    bx0[k] = p.x; bx1[k] = p.x + p.w; by0 = p.y; by1 = p.y + p.h;
  }
  const int dx0 = pl.xdlo[bx0[TBX_MAX_DIGITS - 1]], dx1 = pl.xdhi[bx1[0] - 1], dy0 = pl.ydlo[by0], dy1 = pl.ydhi[by1 - 1];
  const int ncol = dx1 - dx0 + 1, nrow = dy1 - dy0 + 1;
  if (ncol < 1 || ncol > TBX_SC_MAX_COLS || nrow < 1 || nrow > TBX_SC_MAX_ROWS) return;
  std::vector<uint8_t> gray(base0, base0 + (size_t)W * H);
  const uint8_t lum = (uint8_t)A.sc_gray;
  for (int c = 0; c < ncol; c++) {
    const int dx = dx0 + c;
    /* the slots whose boxes the column's real taps read */
    int lo = -1, hi = -1;
    for (int k = 0; k < TBX_MAX_DIGITS; k++) {
      bool touch = false;
      for (int kx = rs.x.start[dx]; kx < rs.x.start[dx + 1]; kx++) touch |= rs.x.si[kx] >= bx0[k] && rs.x.si[kx] < bx1[k];
      if (touch) { if (lo < 0) lo = k; hi = k; }
    }
    if (hi > lo + 1) return; /* three slots under one column: not this table's case */
    A.sc_slot[c] = lo < 0 ? 255 : (uint8_t)lo;
    for (int da = 0; da <= 10; da++)
      for (int db = 0; db <= 10; db++) {
        /* a score that shows digit da in slot lo and db in slot lo + 1 (10: the slot is empty); impossible pairs keep the base */
        bool possible = lo >= 0 && da < 10 && !(db == 10 && da == 0 && lo > 0) && !(db < 10 && lo + 1 >= TBX_MAX_DIGITS);
        long long v = 0;
        if (possible) {
          long long pw = 1;
          for (int i = 0; i < lo; i++) pw *= 10;
          v = da * pw + (db < 10 ? db * pw * 10 : 0);
          if (db == 0) v += pw * 100;                  /* a leading zero needs a digit above it */
          if (v > 2147483647LL) possible = false;
          if (db == 0 && lo + 2 >= TBX_MAX_DIGITS) possible = false;
        }
        if (possible) {
          hd.score = (int32_t)v;
          for (int k = lo; k <= lo + 1 && k < TBX_MAX_DIGITS; k++) {
            const TbxPrim p = si_prim(rec.data(), SI_SLOT_SCORE + k);
            if (p.h <= 0) continue;
            for (int y = p.y; y < p.y + p.h; y++)
              for (int x = p.x; x < p.x + p.w; x++)
                if (tbx_prim_covers(p, HOST_BANK, rec.data(), x, y)) gray[(size_t)y * W + x] = lum;
          }
        }
        for (int r = 0; r < nrow; r++) A.sc_px[c][da][db][r] = area_pixel(gray.data(), W, rs, dx, dy0 + r);
        if (possible)
          for (int y = by0; y < by1; y++) memcpy(&gray[(size_t)y * W + bx0[TBX_MAX_DIGITS - 1]], base0 + (size_t)y * W + bx0[TBX_MAX_DIGITS - 1], (size_t)(bx1[0] - bx0[TBX_MAX_DIGITS - 1]));
      }
  }
  A.sc_dx0 = dx0; A.sc_ncol = ncol; A.sc_dy0 = dy0; A.sc_nrow = nrow;
  A.sc_ok = 1;
}

static int gcd_int(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }
/* Space Invaders: the sprite patch tables and the plain-background map of one output size (tbx_direct.h).  `patches`
 * receives n_sets * py_period * px_period entries (empty when the tables would be too large: n_sets = 0). */
void build_si_direct(const Config &c, const ResizeTab &rs, const TbxAreaPlan &pl, const uint8_t *base0, TbxSiDirect &A, std::vector<TbxSpritePatch> &patches) {
  memset(&A, 0, sizeof A);
  patches.clear();
  const int W = TBX_SI_W, H = TBX_SI_H, dw = pl.dw, dh = pl.dh;
  if (c.game != TBX_SPACE_INVADERS || dw % 4 != 0 || dw > TBX_AREA_MAX_DST || dh > TBX_AREA_MAX_DST || pl.tx > 5 || pl.ty > 4) return;
  A.bg_gray = (int32_t)tbx_luma(SI_COLOR_BLACK);
  /* plain output pixels: every real tap reads background in base frame 0 */
  for (int dy = 0; dy < dh; dy++)
    for (int dx = 0; dx < dw; dx++) {
      bool plain = true;
      for (int ky = rs.y.start[dy]; ky < rs.y.start[dy + 1] && plain; ky++)
        for (int kx = rs.x.start[dx]; kx < rs.x.start[dx + 1]; kx++)
          if (base0[(size_t)rs.y.si[ky] * W + rs.x.si[kx]] != (uint8_t)A.bg_gray) { plain = false; break; }
      if (plain) A.plain[dy][dx >> 5] |= 1u << (dx & 31);
    }
  A.px_period = W / gcd_int(W, dw); A.ox_period = dw / gcd_int(W, dw);
  A.py_period = H / gcd_int(H, dh); A.oy_period = dh / gcd_int(H, dh);
  for (int k = 2; k <= TBX_AREA_MAX_DST; k++) A.inv32[k] = 0xffffffffu / (uint32_t)k + 1u;
  A.inv_px = A.px_period > 1 ? 0xffffffffu / (uint32_t)A.px_period + 1u : 0u;
  A.inv_py = A.py_period > 1 ? 0xffffffffu / (uint32_t)A.py_period + 1u : 0u;
  A.ok = 1;
  build_si_score_strip(rs, pl, base0, A);
  /* the patches rely on the tap tables repeating exactly (start offsets and f32 weights, bit for bit): check, do not assume */
  for (int dx = 0; dx + A.ox_period < dw; dx++) {
    if (pl.xs0[dx + A.ox_period] != pl.xs0[dx] + A.px_period) return;
    for (int t = 0; t < TBX_AREA_MAX_TAPS; t++) if (memcmp(&pl.xalpha[t][dx + A.ox_period], &pl.xalpha[t][dx], sizeof(float)) != 0) return;
  }
  for (int dy = 0; dy + A.oy_period < dh; dy++) {
    if (pl.ys0[dy + A.oy_period] != pl.ys0[dy] + A.py_period) return;
    for (int t = 0; t < TBX_AREA_MAX_TAPS; t++) if (memcmp(&pl.yalpha[t][dy + A.oy_period], &pl.yalpha[t][dy], sizeof(float)) != 0) return;
  }
  /* (sprite, colour) pairs of the draw list's 16-pixel-wide bank sprites at scale 1 (si_prim) */
  struct Set { int off, h; uint32_t color; };
  std::vector<Set> sets;
  for (int k = 0; k < 6; k++) sets.push_back({TBX_BANK_INVADER + 10 * k, SI_ENEMY_H, SI_COLOR_ENEMY});
  sets.push_back({TBX_BANK_BOOM, SI_ENEMY_H, SI_COLOR_ENEMY});
  sets.push_back({TBX_BANK_SHIP, SI_ENEMY_H, SI_COLOR_SHIP});
  sets.push_back({TBX_BANK_BOOM, SI_ENEMY_H, SI_COLOR_SHIP});
  sets.push_back({TBX_BANK_BOOM + 10, SI_ENEMY_H, SI_COLOR_SHIP});
  sets.push_back({TBX_BANK_UFO, SI_UFO_H, SI_COLOR_UFO});
  sets.push_back({TBX_BANK_BOOM + 10, SI_ENEMY_H, SI_COLOR_UFO});
  const size_t n_phase = (size_t)A.px_period * A.py_period;
  if (sets.size() > TBX_SD_MAX_SETS || n_phase * sets.size() * sizeof(TbxSpritePatch) > ((size_t)4 << 20)) return; /* no patches: every entry is evaluated */
  /* a phase must have room: the sprite at (xp, yp), fully inside a frame-sized canvas of background */
  std::vector<uint8_t> canvas((size_t)W * H);
  std::vector<TbxSpritePatch> out(n_phase * sets.size());
  for (size_t s = 0; s < sets.size(); s++) {
    const uint8_t g = (uint8_t)tbx_luma(sets[s].color);
    for (int yp = 0; yp < A.py_period; yp++)
      for (int xp = 0; xp < A.px_period; xp++) {
        /* any position with this phase gives the same patch (that is what the period means); take one inside the frame */
        int x = xp, y = yp;
        while (x + 16 > W) x -= A.px_period;
        while (y + sets[s].h > H) y -= A.py_period;
        if (x < 0 || y < 0) return; /* frame smaller than a period + sprite: no patches */
        std::fill(canvas.begin(), canvas.end(), (uint8_t)A.bg_gray);
        for (int r = 0; r < sets[s].h; r++)
          for (int q = 0; q < 16; q++)
            if ((HOST_BANK[sets[s].off + r] >> (15 - q)) & 1u) canvas[(size_t)(y + r) * W + x + q] = g;
        const int dx0 = pl.xdlo[x], dx1 = pl.xdhi[x + 15], dy0 = pl.ydlo[y], dy1 = pl.ydhi[y + sets[s].h - 1];
        const int w = dx1 - dx0 + 1, h = dy1 - dy0 + 1;
        if (w > TBX_SP_MAX_W || h > TBX_SP_MAX_H) return; /* footprint larger than a patch holds: no patches */
        TbxSpritePatch &P = out[(s * A.py_period + yp) * A.px_period + xp];
        P.w = (uint8_t)w; P.h = (uint8_t)h;
        for (int r = 0; r < h; r++)
          for (int q = 0; q < w; q++) P.px[r * TBX_SP_MAX_W + q] = area_pixel(canvas.data(), W, rs, dx0 + q, dy0 + r);
      }
  }
  A.n_sets = (int32_t)sets.size();
  memset(A.set_lut, 255, sizeof A.set_lut);
  for (size_t s = 0; s < sets.size(); s++) {
    const int idx = sets[s].off >= TBX_BANK_BOOM ? 8 + (sets[s].off - TBX_BANK_BOOM) / 10 : (sets[s].off - TBX_BANK_INVADER) / 10;
    for (int k = 0; k < 4; k++) if (A.set_lut[idx][k] == 255) { A.set_lut[idx][k] = (uint8_t)s; break; }
  }
  for (size_t s = 0; s < sets.size(); s++) { A.set_off[s] = (uint16_t)sets[s].off; A.set_gray[s] = (uint8_t)tbx_luma(sets[s].color); A.set_h[s] = (uint8_t)sets[s].h; }
  patches.swap(out);
}

/* Amidar: look-up tables of the direct kernel for one output size (tbx_direct.h) */
void build_ami_direct(const Config &c, const ResizeTab &rs, const TbxAreaPlan &pl, TbxAmiDirect &A) {
  memset(&A, 0, sizeof A);
  const int W = TBX_AMI_W, H = TBX_AMI_H, dw = pl.dw, dh = pl.dh;
  if (c.game != TBX_AMIDAR || dw % 4 != 0 || dw > TBX_AREA_MAX_DST || dh > TBX_AREA_MAX_DST || pl.tx > 4 || pl.ty > 4) return;
  const AmiCfg &cf = c.ami;
  A.gray[0] = tbx_luma(cf.bg_color); A.gray[1] = tbx_luma(cf.unpainted_color); A.gray[2] = tbx_luma(cf.painted_color); A.gray[3] = tbx_luma(cf.inner_painted_color);
  A.player_gray = tbx_luma(cf.player_color); A.enemy_gray = tbx_luma(cf.enemy_color);
  for (int ty = 0; ty < TBX_AMI_BH; ty++) for (int k = 0; k < 2; k++) A.base_looks[ty][k] = ami_looks_of_tags(cf.board[ty][k]);
  for (int k = 2; k <= TBX_AREA_MAX_DST; k++) A.inv32[k] = 0xffffffffu / (uint32_t)k + 1u;
  memset(A.xcol, 255, sizeof A.xcol);
  memset(A.yrow, 255, sizeof A.yrow);
  const int mx0 = AMI_OFF_X, mx1 = AMI_OFF_X + 4 * TBX_AMI_BW, my0 = AMI_OFF_Y, my1 = AMI_OFF_Y + 5 * TBX_AMI_BH;
  if (mx1 > W || my1 > H) return;
  for (int x = mx0; x < mx1; x++) A.xcol[x] = (uint8_t)((x - mx0) / 4);
  for (int y = my0; y < my1; y++) A.yrow[y] = (uint8_t)((y - my0) / 5);
  std::vector<uint8_t> row(W);
  for (int dx = 0; dx < dw; dx++) {
    int cmin = 255, cmax = -1;
    for (int k = rs.x.start[dx]; k < rs.x.start[dx + 1]; k++) {
      const int cc = A.xcol[rs.x.si[k]];
      if (cc == 255) continue;
      A.wordcols[dx >> 2][cc >> 4] |= 3u << (2 * (cc & 15));
      if (cc < cmin) cmin = cc;
      if (cc > cmax) cmax = cc;
    }
    if (cmax >= 0 && cmax - cmin > 1) return;
    int c0 = cmax < 0 ? 0 : cmin;
    if (c0 > TBX_AMI_BW - 2) c0 = TBX_AMI_BW - 2;
    A.col0[dx] = (uint8_t)c0;
    for (int idx = 0; idx < 16; idx++) {
      std::fill(row.begin(), row.end(), (uint8_t)A.gray[0]);
      for (int j = 0; j < 2; j++) {
        const int look = (idx >> (2 * j)) & 3;
        for (int x = mx0 + 4 * (c0 + j); x < mx0 + 4 * (c0 + j + 1); x++) row[x] = (uint8_t)A.gray[look];
      }
      A.hlut[idx][dx] = hsum_row(row.data(), W, pl, dx);
    }
  }
  A.mdy0 = pl.ydlo[my0]; A.mdy1 = pl.ydhi[my1 - 1];
  for (int dy = 0; dy < dh; dy++) {
    const int nreal = rs.y.start[dy + 1] - rs.y.start[dy];
    for (int k = 0; k < TBX_AREA_MAX_TAPS; k++) {
      if (k >= nreal) { A.ysel[dy][k] = A.ysel[dy][0]; continue; }
      const int r = A.yrow[pl.ys0[dy] + k];
      A.ysel[dy][k] = (uint8_t)r;
      if (r != 255) A.dyrows[dy] |= 1u << r;
    }
  }
  { /* HUD digit rows (score, lives, jumps) lie below the maze */
    std::vector<uint32_t> rec(TBX_WORDS(AmiRec), 0);
    TbxHdr &h = *reinterpret_cast<TbxHdr *>(rec.data());
    h.score = 1999999999; h.lives = 1999999999;
    reinterpret_cast<AmiRec *>(rec.data())->jumps = 1999999999;
    int y0 = H;
    for (int s = AMI_SLOT_SCORE; s < AMI_N_SLOTS; s++) { const TbxPrim p = ami_prim(rec.data(), cf, 0, s); if (p.h > 0 && p.y < y0) y0 = p.y; }
    if (y0 < 0) y0 = 0;
    A.hud_dylo = y0 < H ? pl.ydlo[y0] : dh;
    if (A.hud_dylo <= A.mdy1) return;
  }
  A.ok = 1;
}

} /* namespace tbx */
