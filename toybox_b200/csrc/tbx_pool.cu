/* tbx_pool.cu -- the C ABI of include/toybox_b200.h: pool life cycle, launches, JSON import/export. */
#include "../../include/toybox_b200.h"
#include "tbx_kernels.cuh"
#include "tbx_wrap.cuh"
#include "tbx_snapshot.cuh"
#include "tbx_fields.h"
#include "tbx_direct_launch.h"
#include <cmath>
#include <map>
#include <memory>
#include <new>
#include <string>
#include <string.h>
#include <algorithm>
#include <thread>
#include <tuple>
#include <vector>

using namespace tbxk;
using tbxjson::Value;

static thread_local std::string g_err;
static int set_err(int code, const std::string &msg) { g_err = msg; return code; }
#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess) return set_err(TBX_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

/* f() with every exception turned into an error code: nothing may unwind through the C ABI into the caller */
template <class F> static int guarded(F &&f) {
  try {
    return f();
  } catch (const std::bad_alloc &) {
    return set_err(TBX_ENOMEM, "out of host memory");
  } catch (const std::exception &e) {
    return set_err(TBX_EJSON, e.what());
  }
}

/* render resources of one INTER_AREA output size: the plan, then those of each layout, built on its first render */
struct AreaRes {
  TbxAreaPlan plan;
  Buf<TbxAreaPlan> d_plan;
  Buf<uint8_t> d_base_out[2];       /* gray: down-samples of base frames 0/1 */
  Buf<TbxDigitPatch> d_patches[2];
  Buf<uint8_t> d_direct, d_direct2; /* tables of the direct kernel (tbx_direct.h), empty when the pair is not covered */
  Buf<uint8_t> d_rgb_out[2];        /* RGB: interleaved down-samples of base frames 0/1 */
};
/* base frames 0/1 of the current config (see tbx_render.cuh): gray, RGBA and packed RGB on the device, gray on the host;
 * for the RGB INTER_AREA layout also R, G, B planes of W x H each (the tile kernel reads one channel's source window in
 * 4-byte words), on the device and the host, built on the first such render */
struct BaseFrames {
  Buf<uint8_t> gray[2], rgba[2], rgb[2], planar[2];
  std::vector<uint8_t> h_gray[2], h_planar[2];
};
/* tbx_step_host's stream and staging */
struct HostStaging {
  cudaStream_t s = 0;
  Buf<int32_t> actions, reward, score, lives;
  Buf<uint8_t> done, obs;
  ~HostStaging() { if (s) cudaStreamDestroy(s); }
};

/* a pool's interned geometry tables, per game: std::get<GAME>(tbx_pool::tabs); Space Invaders has none */
template <int G> using Tables = std::vector<typename Traits<G>::Table>;
template <int G> static constexpr bool kTables = G != TBX_SPACE_INVADERS;
static_assert(TBX_BREAKOUT == 0 && TBX_AMIDAR == 1 && TBX_SPACE_INVADERS == 2, "game ids index tbx_pool::tabs");

struct tbx_pool {
  int game, n, n_pad, device;
  const tbx::GameInfo *info;
  tbx::Config cfg;
  Buf<uint8_t> d_cfg;
  std::tuple<Tables<TBX_BREAKOUT>, Tables<TBX_AMIDAR>, Tables<TBX_SPACE_INVADERS>> tabs;
  Buf<uint8_t> d_tables;
  int d_tables_n;
  Buf<uint32_t> planes;
  Buf<unsigned long long> d_stats;
  Buf<int> d_bad; /* [0] = invalid action ids, [1] = skipped snapshot entries, since the last tbx_check */
  Buf<int32_t> d_legal;
  /* render resources of the current config: base frames, and per output size the INTER_AREA plan */
  std::unique_ptr<BaseFrames> base;
  std::map<std::pair<int, int>, AreaRes> area;
  Buf<int32_t> d_dense; /* [0] = count, [8..] = env ids the patch kernel left to the canvas kernel */
  Buf<int32_t> d_fb;    /* [0] = count, [1] = finished CTAs, [8..] = env ids the direct INTER_AREA kernel left to the tile kernel */
  /* JSON import / export staging (grown on demand, kept): env ids and AoS records on the device, records in pinned host memory */
  Buf<int32_t> j_ids;
  Buf<uint32_t> j_recs;
  PinnedBuf<uint32_t> j_host;
  std::unique_ptr<HostStaging> hs;
  /* snapshot loads: owner entry per env (duplicate destinations), blob -> pool table indices (foreign tables) */
  Buf<int32_t> d_owner, d_remap;
};

template <int G, class P> static auto &tables(P *p) { return std::get<G>(p->tabs); }
/* the game's part of a config */
template <int G, class C> static auto &game_cfg(C &c) {
  if constexpr (G == TBX_BREAKOUT) return c.brk;
  else if constexpr (G == TBX_AMIDAR) return c.ami;
  else return c.si;
}
static uint64_t *cfg_rand(tbx::Config &c) { return with_game(c.game, [&](auto g) { return game_cfg<decltype(g)::value>(c).rand; }); }
/* Breakout's default brick table (the base frames show its bricks); NULL for the other games */
static const BrkTable *brk_default(const tbx_pool *p) { return p->game == TBX_BREAKOUT ? &tables<TBX_BREAKOUT>(p)[p->cfg.brk.default_tbl] : 0; }

/* per-game host codecs, overloaded on the game's record and table types */
static void fit_table(const tbx::Config &c, BrkTable &t) { tbx::brk_mark_delta_ok(c, t); } /* delta_ok depends on the config */
static void fit_table(const tbx::Config &, AmiTable &) {}
static void default_table(const tbx::Config &c, BrkTable &t) { tbx::brk_default_table(c.brk, t); fit_table(c, t); }
static void default_table(const tbx::Config &c, AmiTable &t) { tbx::ami_default_table(c.ami, t); }
static Value state_to_json(const BrkRec &r, const BrkTable *t) { return tbx::brk_state_to_json(r, *t); }
static Value state_to_json(const AmiRec &r, const AmiTable *t) { return tbx::ami_state_to_json(r, *t); }
static Value state_to_json(const SiRec &r, const int *) { return tbx::si_state_to_json(r); }
static void state_from_json(const Value &v, BrkRec &r, BrkTable &t) { tbx::brk_state_from_json(v, r, t); }
static void state_from_json(const Value &v, AmiRec &r, AmiTable &t) { tbx::ami_state_from_json(v, r, t); }

/* The JSON codec is host work per env (build / walk a document tree, print / parse ~20-40 KB of text): spread the envs of a
 * batched call over host threads.  f(i) may throw; the first message is re-thrown on the calling thread. */
template <class F> static void parallel_for(int n, F f) {
  int nt = (int)std::thread::hardware_concurrency();
  if (const char *env = getenv("TBX_JSON_THREADS")) nt = atoi(env);
  nt = std::max(1, std::min(std::min(nt, 32), n / 8));
  if (nt <= 1) { for (int i = 0; i < n; i++) f(i); return; }
  std::vector<std::string> errs(nt);
  std::vector<std::thread> th;
  for (int t = 0; t < nt; t++)
    th.emplace_back([&, t]() {
      try { for (int i = t; i < n; i += nt) f(i); } catch (const std::exception &e) { errs[t] = e.what(); if (errs[t].empty()) errs[t] = "error"; }
    });
  for (auto &x : th) x.join();
  for (auto &e : errs) if (!e.empty()) throw std::runtime_error(e);
}

static int blocks(int n, int t) { return (n + t - 1) / t; }

static int upload_cfg(tbx_pool *p) {
  return with_game(p->game, [&](auto g) -> int {
    const auto &c = game_cfg<decltype(g)::value>(p->cfg);
    CK(p->d_cfg.grow(sizeof c));
    CK(cudaMemcpy(p->d_cfg, &c, sizeof c, cudaMemcpyHostToDevice));
    return TBX_OK;
  });
}
static int upload_tables(tbx_pool *p) {
  return with_game(p->game, [&](auto g) -> int {
    const auto &t = tables<decltype(g)::value>(p);
    if (t.empty() || (int)t.size() == p->d_tables_n) return TBX_OK;
    CK(cudaDeviceSynchronize());
    Buf<uint8_t> d;
    CK(d.upload(reinterpret_cast<const uint8_t *>(t.data()), t.size() * sizeof t[0]));
    p->d_tables = std::move(d);
    p->d_tables_n = (int)t.size();
    return TBX_OK;
  });
}
/* index of an identical table, appending it if new */
template <class TT> static int intern(std::vector<TT> &v, const TT &t) {
  for (size_t i = 0; i < v.size(); i++) if (memcmp(&v[i], &t, sizeof t) == 0) return (int)i;
  v.push_back(t);
  return (int)v.size() - 1;
}
static void install_default_table(tbx_pool *p) {
  with_game(p->game, [&](auto g) {
    constexpr int G = decltype(g)::value;
    if constexpr (kTables<G>) {
      typename Traits<G>::Table t;
      default_table(p->cfg, t);
      game_cfg<G>(p->cfg).default_tbl = intern(tables<G>(p), t);
    }
  });
}

template <int GAME> static int launch_step(tbx_pool *p, const StepArgs &a, cudaStream_t s) {
  /* staged (records through shared memory) where it measures faster; TBX_STEP_STAGED=0/1 overrides (tuning, tests) */
  bool staged = GAME == TBX_SPACE_INVADERS; /* measured, 65,536 envs in steady state: Space Invaders 90 vs 178 us; Breakout 39 vs 37; Amidar 69 vs 61 */
  if (const char *env = getenv("TBX_STEP_STAGED")) staged = atoi(env) != 0;
  if (staged) {
    constexpr int EPB = StepGeom<GAME>::EPB, smem = Traits<GAME>::RW * EPB * 4;
    CK((cudaFuncSetAttribute(step_staged_kernel<GAME>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
    step_staged_kernel<GAME><<<blocks(p->n, EPB), EPB, smem, s>>>(a);
  } else {
    step_kernel<GAME><<<blocks(p->n, 128), 128, 0, s>>>(a);
  }
  CK(cudaGetLastError());
  return TBX_OK;
}
static int do_new_game(tbx_pool *p, const uint8_t *mask, cudaStream_t s) {
  with_game(p->game, [&](auto g) {
    new_game_kernel<decltype(g)::value><<<blocks(p->n, 128), 128, 0, s>>>(p->planes, p->n, p->n_pad, p->d_cfg, p->d_tables, mask);
  });
  CK(cudaGetLastError());
  return TBX_OK;
}

/* device side of tbx_pool_create */
static int init_device(tbx_pool *p) {
  const size_t plane_words = (size_t)p->info->rec_words * p->n_pad;
  CK(cudaSetDevice(p->device));
  CK(p->planes.alloc(plane_words));
  CK(cudaMemset(p->planes, 0, plane_words * sizeof(uint32_t)));
  CK(p->d_stats.alloc(4));
  CK(cudaMemset(p->d_stats, 0, 4 * sizeof(unsigned long long)));
  CK(p->d_bad.alloc(2));
  CK(cudaMemset(p->d_bad, 0, 2 * sizeof(int)));
  CK(p->d_legal.upload(p->info->legal, 18));
  int r = upload_cfg(p);
  if (r) return r;
  r = upload_tables(p);
  if (r) return r;
  const uint64_t *rand = cfg_rand(p->cfg);
  set_sim_rand_kernel<<<blocks(p->n, 256), 256>>>(p->planes, p->n, p->n_pad, rand[0], rand[1]);
  CK(cudaGetLastError());
  for (int k = 0; k < p->info->new_games_at_ctor; k++) { r = do_new_game(p, 0, 0); if (r) return r; }
  CK(cudaDeviceSynchronize());
  return TBX_OK;
}

extern "C" {

const char *tbx_last_error(void) { return g_err.c_str(); }
int tbx_version(void) { return 100; }

int tbx_pool_destroy(tbx_pool *p) {
  if (!p) return TBX_OK;
  cudaSetDevice(p->device);
  cudaDeviceSynchronize();
  delete p;
  return TBX_OK;
}

int tbx_pool_create(const char *game, int n_envs, int device, const char *cfg_json, tbx_pool **out) {
  if (!out) return set_err(TBX_EINVAL, "out is NULL");
  *out = 0;
  int g = tbx::game_from_name(game);
  if (g < 0) return set_err(TBX_EINVAL, std::string("unknown game '") + (game ? game : "(null)") + "'");
  if (n_envs < 1) return set_err(TBX_EINVAL, "n_envs must be >= 1");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
    return set_err(TBX_ECUDA, "no CUDA device available: toybox_b200 has no CPU path");
  if (device < 0 || device >= ndev) return set_err(TBX_EINVAL, "device index out of range");
  return guarded([&]() -> int {
    std::unique_ptr<tbx_pool> p(new tbx_pool());
    p->game = g; p->n = n_envs; p->n_pad = (n_envs + 31) & ~31; p->device = device; p->info = tbx::game_info(g);
    tbx::default_config(g, p->cfg);
    if (cfg_json) tbx::config_from_json(p->cfg, tbxjson::parse(cfg_json));
    install_default_table(p.get());
    const int rc = init_device(p.get());
    if (rc) { std::string keep = g_err; tbx_pool_destroy(p.release()); g_err = keep; return rc; }
    *out = p.release();
    return TBX_OK;
  });
}

int tbx_frame_width(const tbx_pool *p) { return p ? p->info->width : 0; }
int tbx_frame_height(const tbx_pool *p) { return p ? p->info->height : 0; }
int tbx_n_envs(const tbx_pool *p) { return p ? p->n : 0; }
int tbx_device(const tbx_pool *p) { return p ? p->device : -1; }
int tbx_legal_actions(const tbx_pool *p, int32_t *out, int cap) {
  if (!p) return 0;
  for (int i = 0; i < p->info->n_legal && i < cap; i++) out[i] = p->info->legal[i];
  return p->info->n_legal;
}
size_t tbx_obs_bytes(const tbx_pool *p, int mode, int out_w, int out_h) {
  if (!p) return 0;
  size_t px = (size_t)p->info->width * p->info->height;
  switch (mode) {
    case TBX_OBS_RGBA: return px * 4;
    case TBX_OBS_RGB: return px * 3;
    case TBX_OBS_GRAY: return px;
    case TBX_OBS_GRAY_AREA:
    case TBX_OBS_RGB_AREA:
      if (out_w < 1 || out_h < 1 || out_w > p->info->width || out_h > p->info->height || out_w > TBX_RS_MAX_DST || out_h > TBX_RS_MAX_DST) return 0;
      return (size_t)out_w * out_h * (mode == TBX_OBS_RGB_AREA ? 3 : 1);
  }
  return 0;
}

int tbx_seed(tbx_pool *p, const uint32_t *seeds, const int32_t *ids, int n) {
  if (!p || !seeds || n < 0) return set_err(TBX_EINVAL, "bad arguments");
  if (!ids && n > p->n) return set_err(TBX_EINVAL, "more seeds than envs");
  if (n == 0) return TBX_OK;
  if (ids) for (int i = 0; i < n; i++) if (ids[i] < 0 || ids[i] >= p->n) return set_err(TBX_EINVAL, "env id out of range");
  CK(cudaSetDevice(p->device));
  Buf<uint32_t> d_seeds;
  Buf<int32_t> d_ids;
  CK(d_seeds.upload(seeds, n));
  if (ids) CK(d_ids.upload(ids, n));
  seed_kernel<<<blocks(n, 256), 256>>>(p->planes, p->n_pad, d_seeds, d_ids, n);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return TBX_OK;
}

int tbx_new_game(tbx_pool *p, const uint8_t *mask, void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  CK(cudaSetDevice(p->device));
  return do_new_game(p, mask, (cudaStream_t)stream);
}

struct SynStream { uint64_t seed, env0, t; };
static int do_step(tbx_pool *p, const int32_t *actions, const uint8_t *inputs, int auto_reset, int32_t *reward, uint8_t *done,
                   int32_t *score, int32_t *lives, cudaStream_t s, const SynStream *syn = 0) {
  StepArgs a;
  a.planes = p->planes; a.n = p->n; a.n_pad = p->n_pad; a.cfg = p->d_cfg; a.tables = p->d_tables;
  a.actions = actions; a.inputs = inputs; a.auto_reset = auto_reset;
  a.legal = p->d_legal; a.n_legal = p->info->n_legal;
  a.syn_seed = syn ? syn->seed : 0; a.syn_env0 = syn ? syn->env0 : 0; a.syn_t = syn ? syn->t : 0;
  a.reward = reward; a.done = done; a.score = score; a.lives = lives; a.stats = p->d_stats; a.bad_actions = p->d_bad;
  return with_game(p->game, [&](auto g) { return launch_step<decltype(g)::value>(p, a, s); });
}
int tbx_step(tbx_pool *p, const int32_t *actions, int auto_reset, int32_t *reward, uint8_t *done, int32_t *score, int32_t *lives, void *stream) {
  if (!p || !actions) return set_err(TBX_EINVAL, "pool/actions is NULL");
  CK(cudaSetDevice(p->device));
  return do_step(p, actions, 0, auto_reset, reward, done, score, lives, (cudaStream_t)stream);
}
int tbx_step_random(tbx_pool *p, uint64_t seed, uint64_t env0, uint64_t t, int auto_reset, int32_t *reward, uint8_t *done, int32_t *score, int32_t *lives,
                    void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  CK(cudaSetDevice(p->device));
  SynStream syn = {seed, env0, t};
  return do_step(p, 0, 0, auto_reset, reward, done, score, lives, (cudaStream_t)stream, &syn);
}
int tbx_step_inputs(tbx_pool *p, const uint8_t *inputs, int auto_reset, int32_t *reward, uint8_t *done, int32_t *score, int32_t *lives, void *stream) {
  if (!p || !inputs) return set_err(TBX_EINVAL, "pool/inputs is NULL");
  CK(cudaSetDevice(p->device));
  return do_step(p, 0, inputs, auto_reset, reward, done, score, lives, (cudaStream_t)stream);
}
int tbx_check(tbx_pool *p, void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  CK(cudaSetDevice(p->device));
  int bad[2] = {0, 0};
  CK(cudaMemcpyAsync(bad, p->d_bad, sizeof bad, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  if (bad[0]) {
    CK(cudaMemsetAsync(p->d_bad, 0, sizeof(int), (cudaStream_t)stream));
    return set_err(TBX_EACTION, "Expected to apply action, but failed: " + std::to_string(bad[0]) + " invalid ALE action id(s)");
  }
  if (bad[1]) {
    CK(cudaMemsetAsync(p->d_bad + 1, 0, sizeof(int), (cudaStream_t)stream));
    return set_err(TBX_EINVAL, "state snapshot: " + std::to_string(bad[1]) + " entr" + (bad[1] == 1 ? "y" : "ies") +
                                   " skipped (env id, column or table index out of range)");
  }
  return TBX_OK;
}

} /* extern "C" */

/* ---- render */
static void drop_render_cache(tbx_pool *p) {
  p->base.reset();
  p->area.clear();
}
/* base frames 0/1 of the current config (see tbx_render.cuh); kept only once every buffer is in place */
static int ensure_base(tbx_pool *p) {
  if (p->base) return TBX_OK;
  auto base = std::make_unique<BaseFrames>();
  const int npix = p->info->width * p->info->height;
  std::vector<uint32_t> rgba(npix);
  std::vector<uint8_t> rgb((size_t)npix * 3);
  for (int b = 0; b < 2; b++) {
    std::vector<uint8_t> &gray = base->h_gray[b];
    gray.resize(npix);
    tbx::build_base_frame(p->cfg, brk_default(p), b, rgba.data());
    tbx::frame_to_gray(rgba.data(), npix, gray.data());
    CK(base->gray[b].alloc(npix + 16)); /* slack: the direct kernel reads whole words around a pixel */
    CK(cudaMemset(base->gray[b] + npix, 0, 16));
    CK(cudaMemcpy(base->gray[b], gray.data(), npix, cudaMemcpyHostToDevice));
    CK(base->rgba[b].upload(reinterpret_cast<const uint8_t *>(rgba.data()), (size_t)npix * 4));
    for (int i = 0; i < npix; i++) { uint32_t c = rgba[i]; rgb[3 * i] = c & 255; rgb[3 * i + 1] = (c >> 8) & 255; rgb[3 * i + 2] = (c >> 16) & 255; }
    CK(base->rgb[b].upload(rgb.data(), rgb.size()));
  }
  p->base = std::move(base);
  return TBX_OK;
}
/* base frames 0/1 as planes for the RGB INTER_AREA layout; kept only once both are in place */
static int ensure_planar(tbx_pool *p) {
  BaseFrames &bf = *p->base;
  if (bf.planar[0]) return TBX_OK;
  const int npix = p->info->width * p->info->height;
  std::vector<uint32_t> rgba(npix);
  std::vector<uint8_t> h[2];
  Buf<uint8_t> d[2];
  for (int b = 0; b < 2; b++) {
    tbx::build_base_frame(p->cfg, brk_default(p), b, rgba.data());
    h[b].resize((size_t)npix * 3);
    for (int c = 0; c < 3; c++)
      for (int i = 0; i < npix; i++) h[b][(size_t)c * npix + i] = (uint8_t)(rgba[i] >> (8 * c));
    CK(d[b].upload(h[b].data(), h[b].size()));
  }
  for (int b = 0; b < 2; b++) { bf.planar[b] = std::move(d[b]); bf.h_planar[b] = std::move(h[b]); }
  return TBX_OK;
}
/* the INTER_AREA resources of one output size and layout, built on first use; each part is kept only once every buffer
 * of it is in place */
static int ensure_area(tbx_pool *p, int out_w, int out_h, bool rgb, const AreaRes **out) {
  auto key = std::make_pair(out_w, out_h);
  auto it = p->area.find(key);
  if (it != p->area.end() && (rgb ? it->second.d_rgb_out[0] : it->second.d_base_out[0])) { *out = &it->second; return TBX_OK; }
  tbx::ResizeTab rs;
  try { tbx::build_resize(p->info->width, p->info->height, out_w, out_h, rs); }
  catch (const std::exception &e) { return set_err(TBX_EINVAL, e.what()); }
  if (it == p->area.end()) {
    AreaRes r;
    if (!tbx::build_area_plan(rs, r.plan)) return set_err(TBX_EINVAL, "resize: the fused kernel supports destinations up to 128x128 with at most 8 taps per axis");
    CK(r.d_plan.upload(&r.plan, 1));
    it = p->area.emplace(key, std::move(r)).first;
  }
  AreaRes &ar = it->second;
  if (!rgb && !ar.d_base_out[0]) {
    Buf<uint8_t> base_out[2], direct, direct2;
    Buf<TbxDigitPatch> patches[2];
    for (int b = 0; b < 2; b++) {
      const uint8_t *gray = p->base->h_gray[b].data();
      std::vector<uint8_t> h(((size_t)out_w * out_h + 15) & ~(size_t)15, 0);
      tbx::area_resize(gray, rs, h.data());
      CK(base_out[b].upload(h.data(), h.size()));
      std::vector<TbxDigitPatch> hp((size_t)TBX_DP_SLOTS * 10);
      tbx::build_digit_patches(p->cfg, brk_default(p), rs, ar.plan, gray, hp.data());
      CK(patches[b].upload(hp.data(), hp.size()));
    }
    CK(tbx_direct_build(p->cfg, brk_default(p), rs, ar.plan, p->base->h_gray[0].data(), direct, direct2));
    for (int b = 0; b < 2; b++) { ar.d_base_out[b] = std::move(base_out[b]); ar.d_patches[b] = std::move(patches[b]); }
    ar.d_direct = std::move(direct); ar.d_direct2 = std::move(direct2);
  }
  if (rgb && !ar.d_rgb_out[0]) { /* the per-channel resize of the planar base frames, interleaved */
    int r = ensure_planar(p);
    if (r) return r;
    const size_t npix = (size_t)p->info->width * p->info->height, nout = (size_t)out_w * out_h;
    Buf<uint8_t> rgb_out[2];
    std::vector<uint8_t> plane(nout), h((nout * 3 + 15) & ~(size_t)15, 0);
    for (int b = 0; b < 2; b++) {
      for (int c = 0; c < 3; c++) {
        tbx::area_resize(p->base->h_planar[b].data() + c * npix, rs, plane.data());
        for (size_t i = 0; i < nout; i++) h[3 * i + c] = plane[i];
      }
      CK(rgb_out[b].upload(h.data(), h.size()));
    }
    for (int b = 0; b < 2; b++) ar.d_rgb_out[b] = std::move(rgb_out[b]);
  }
  *out = &ar;
  return TBX_OK;
}

static int align16(int v) { return (v + 15) & ~15; }
/* canvas bytes per pixel of an observation layout */
static constexpr int obs_pix(int mode) { return mode == TBX_OBS_RGBA ? 4 : mode == TBX_OBS_RGB ? 3 : 1; }
/* f(Const<MODE>()) for a native layout */
template <class F> static int with_layout(int mode, F &&f) {
  if (mode == TBX_OBS_RGBA) return f(Const<TBX_OBS_RGBA>());
  if (mode == TBX_OBS_RGB) return f(Const<TBX_OBS_RGB>());
  return f(Const<TBX_OBS_GRAY>());
}

/* the canvas kernel (tbx_render.cuh): the dense Breakout / Amidar envs the patch kernel lists */
template <int GAME, int MODE> static int launch_render(const RenderArgs &a, const typename Traits<GAME>::Cfg &cfg, int smem, cudaStream_t s) {
  /* the opt-in is per device (a process may hold pools on several GPUs): set it on every launch, a cheap host-side call */
  CK((cudaFuncSetAttribute(render_kernel<GAME, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem > 160 * 1024 ? smem : 160 * 1024)));
  const int H = Traits<GAME>::H;
  dim3 grid(blocks(a.n, TBX_EPC), (H + a.band_rows - 1) / a.band_rows);
  /* measured: Breakout's few primitives keep 4 warps busy, the sprite-heavy games use 8 (profiles/r1_native_layouts.md) */
  const int threads = GAME == TBX_BREAKOUT ? 128 : 256;
  render_kernel<GAME, MODE><<<grid, threads, smem, s>>>(a, cfg);
  CK(cudaGetLastError());
  return TBX_OK;
}
/* native layouts as broadcast + patch (tbx_render_native.cuh) */
template <int GAME, int PIX> static int launch_native(const RenderArgs &a, const typename Traits<GAME>::Cfg &cfg, int band_smem, cudaStream_t s) {
  const int threads = 256;
  const int patch_smem = a.smem_canvas; /* the records of the CTA's 8 envs */
  CK((cudaFuncSetAttribute(base_fill_kernel<GAME, PIX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024)));
  CK((cudaFuncSetAttribute(native_patch_kernel<GAME, PIX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024)));
  if (band_smem > 64 * 1024 || patch_smem > 160 * 1024) return set_err(TBX_EINVAL, "frame too wide for the native render path");
  const int H = Traits<GAME>::H;
  dim3 grid(blocks(a.n, TBX_FILL_ENVS), (H + a.band_rows - 1) / a.band_rows);
  base_fill_kernel<GAME, PIX><<<grid, 128, band_smem, s>>>(a, cfg);
  CK(cudaGetLastError());
  native_patch_kernel<GAME, PIX><<<blocks(a.n, TBX_EPC), threads, patch_smem, s>>>(a, cfg);
  CK(cudaGetLastError());
  return TBX_OK;
}
/* INTER_AREA, one warp per env (tbx_render_area.cuh); RGB: the RGB mode */
template <int GAME, int TX, int TY, bool DUAL, bool RGB = false>
static int launch_area_tile(const RenderArgs &a, const typename Traits<GAME>::Cfg &cfg, const TbxAreaPlan &plan, int smem, cudaStream_t s) {
  CK((cudaFuncSetAttribute(area_tile_kernel<GAME, TX, TY, DUAL, RGB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
  /* env-list mode (the envs the direct kernel handed over, normally none): a small grid walks the list */
  const int grid = a.env_list ? (blocks(a.n, TBX_EPC) < 296 ? blocks(a.n, TBX_EPC) : 296) : blocks(a.n, TBX_EPC);
  area_tile_kernel<GAME, TX, TY, DUAL, RGB><<<grid, TBX_TILE_THREADS, smem, s>>>(a, cfg, plan);
  CK(cudaGetLastError());
  return TBX_OK;
}

/* INTER_AREA: the direct kernel where it covers the pair, then the tile kernel; RGB: the tile kernel's RGB mode alone (single
 * frames, and the wrapped path's max of two frames) */
static int render_area(tbx_pool *p, RenderArgs &a, int out_w, int out_h, bool rgb, cudaStream_t s) {
  const AreaRes *ar = 0;
  int r = ensure_area(p, out_w, out_h, rgb, &ar);
  if (r) return r;
  const TbxAreaPlan &plan = ar->plan;
  const bool dual = a.planes2 != 0;
  a.plan = ar->d_plan;
  if (rgb) {
    for (int b = 0; b < 2; b++) { a.base[b] = p->base->planar[b]; a.base_out[b] = ar->d_rgb_out[b]; a.patches[b] = 0; }
  } else {
    a.base_out[0] = ar->d_base_out[0]; a.base_out[1] = ar->d_base_out[1];
    const char *env = getenv("TBX_AREA_DIGIT_CACHE");
    const bool on = !(env && atoi(env) == 0);
    a.patches[0] = on ? ar->d_patches[0].get() : 0; a.patches[1] = on ? ar->d_patches[1].get() : 0;
  }
  const Taps taps = inst_taps(plan.tx, plan.ty);
  if (dual && taps.x == 8) return set_err(TBX_EINVAL, "wrapped observations need an output size the tile kernel supports (at most 5 x 4 taps)");
  /* one warp per env over tiles of 16 x 8 output pixels, runs of at most TBX_TILE_MAX_RUN tiles: the scratch holds the
   * widest / tallest run window of the instantiated tap counts */
  const int tile_h = 1 << TBX_TILE_HSHIFT;
  int stride = 0, rows = 0;
  for (int dxA = 0; dxA < out_w; dxA += 16) {
    const int dxL = dxA + 16 * TBX_TILE_MAX_RUN - 1 < out_w ? dxA + 16 * TBX_TILE_MAX_RUN - 1 : out_w - 1;
    const int wdt = ((plan.xs0[dxL] + taps.x + 3) & ~3) - (plan.xs0[dxA] & ~3);
    if (wdt > stride) stride = wdt;
  }
  for (int dyA = 0; dyA < out_h; dyA += tile_h) {
    const int dyL = dyA + tile_h - 1 < out_h ? dyA + tile_h - 1 : out_h - 1;
    const int rws = plan.ys0[dyL] + taps.y - plan.ys0[dyA];
    if (rws > rows) rows = rws;
  }
  /* every plan build_area_plan accepts fits, for all three games (at most 256 B x 64 rows) */
  if (stride > 512 || rows > 96 || p->info->width % 4 != 0)
    return set_err(TBX_EINVAL, "INTER_AREA " + std::to_string(out_w) + "x" + std::to_string(out_h) + ": the tile kernel's scratch window (" +
                                   std::to_string(stride) + " B x " + std::to_string(rows) + " rows) exceeds its limit of 512 B x 96 rows");
  a.tile_stride = stride;
  a.list_cap = TBX_TILE_LCAP;
  if (const char *env = getenv("TBX_AREA_LCAP")) a.list_cap = atoi(env); /* tests: small lists force the sweep / per-tile paths */
  if (a.list_cap < 1 || a.list_cap > TBX_TILE_LCAP) a.list_cap = TBX_TILE_LCAP;
  a.tile_bytes = align16(stride * rows);
  a.warp_bytes = TBX_TILE_LCAP * (rgb ? 24 : 20) + 32 + a.tile_bytes * (dual ? 2 : 1); /* list, extents (, colours), tile mask, scratch */
  const int smem = a.smem_canvas + (TBX_TILE_THREADS / 32) * a.warp_bytes;
  int smem_optin = 0;
  CK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device));
  if (smem > smem_optin)
    return set_err(TBX_EINVAL, "INTER_AREA " + std::to_string(out_w) + "x" + std::to_string(out_h) + ": the tile kernel needs " + std::to_string(smem) +
                                   " B of shared memory per CTA, the device allows " + std::to_string(smem_optin));
  /* Direct kernel first (tbx_render_direct.cuh; TBX_AREA_KERNEL=tile turns it off): closed forms for the envs they
   * cover, the rest are listed and rendered by the tile kernel in env-list mode right after (usually an empty list) */
  const char *ksel = getenv("TBX_AREA_KERNEL");
  if (ar->d_direct && !dual && !rgb && !(ksel && !strcmp(ksel, "tile"))) {
    if (!p->d_fb) { /* the counters start at zero; the kernels leave them so */
      Buf<int32_t> fb;
      CK(fb.alloc((size_t)p->n_pad + 8));
      CK(cudaMemsetAsync(fb, 0, 8 * sizeof(int32_t), s));
      p->d_fb = std::move(fb);
    }
    DirectArgs da = {};
    da.aux = ar->d_direct; da.aux2 = ar->d_direct2; da.fb_list = p->d_fb + 8; da.fb_count = p->d_fb; da.sched = p->d_fb + 2;
    CK(tbx_launch_direct(p->cfg, a, plan, da, s));
    if (p->game == TBX_SPACE_INVADERS) return TBX_OK; /* covers every env: nothing is handed over */
    a.env_list = p->d_fb + 8;
    a.env_count = p->d_fb;
  }
  return with_game(p->game, [&](auto g) {
    constexpr int G = decltype(g)::value;
    const auto &cfg = game_cfg<G>(p->cfg);
    return with_taps<8>(plan.tx, plan.ty, [&](auto X, auto Y) {
      constexpr int TX = decltype(X)::value, TY = decltype(Y)::value;
      if constexpr (TX == 8) { /* single frames only (checked above) */
        return rgb ? launch_area_tile<G, 8, 8, false, true>(a, cfg, plan, smem, s) : launch_area_tile<G, 8, 8, false>(a, cfg, plan, smem, s);
      } else if (rgb) {
        return dual ? launch_area_tile<G, TX, TY, true, true>(a, cfg, plan, smem, s) : launch_area_tile<G, TX, TY, false, true>(a, cfg, plan, smem, s);
      } else {
        return dual ? launch_area_tile<G, TX, TY, true>(a, cfg, plan, smem, s) : launch_area_tile<G, TX, TY, false>(a, cfg, plan, smem, s);
      }
    });
  });
}

/* Native layouts: broadcast + patch (tbx_render_native.cuh) -- the base frame leaves through the TMA engine at HBM speed,
 * what differs from it is painted straight into the frame.  Breakout and Amidar envs that differ in many places (a wall
 * with more than 20 holes, a maze with more than 48 painted tiles / boxes; TBX_NATIVE_DENSE overrides) are cheaper to
 * repaint in shared memory: the patch kernel lists them and the canvas kernel below renders exactly those.  Space
 * Invaders' ~50 sprites are always patched. */
static int render_native(tbx_pool *p, RenderArgs &a, int mode, cudaStream_t s) {
  const int W = p->info->width, H = p->info->height, pix = obs_pix(mode);
  /* canvas bands of at most ~40 KB so that five CTAs stay resident per SM */
  int max_rows = (40 * 1024) / (W * pix);
  if (max_rows < 1) max_rows = 1;
  const int nb = (H + max_rows - 1) / max_rows;
  a.band_rows = (H + nb - 1) / nb;
  a.smem_rects = a.smem_canvas + align16(a.band_rows * W * pix);
  const int smem_total = a.smem_rects + 2 * TBX_MAX_RECTS * (int)sizeof(int4) + 128 + TBX_MAX_BIG * (int)sizeof(uint4); /* + list counts, per-env base / env ids, the big-primitive queue */
  if (smem_total > 220 * 1024) return set_err(TBX_EINVAL, "observation size needs more shared memory than one SM has");
  return with_game(p->game, [&](auto g) -> int {
    constexpr int G = decltype(g)::value;
    const auto &cfg = game_cfg<G>(p->cfg);
    auto patch = [&]() { return with_layout(mode, [&](auto m) { return launch_native<G, obs_pix(decltype(m)::value)>(a, cfg, align16(a.band_rows * W * pix), s); }); };
    if constexpr (G == TBX_SPACE_INVADERS) {
      return patch();
    } else {
      int thr = G == TBX_BREAKOUT ? 20 : 48;
      if (const char *dense_env = getenv("TBX_NATIVE_DENSE")) thr = atoi(dense_env) < 0 ? INT32_MAX : atoi(dense_env);
      if (thr != INT32_MAX) {
        CK(p->d_dense.grow((size_t)p->n_pad + 8 + p->n_pad / 4)); /* + a byte per env */
        a.dense_list = p->d_dense + 8;
        a.dense_count = p->d_dense;
        a.dense_flag = reinterpret_cast<uint8_t *>(p->d_dense + 8 + p->n_pad);
        a.dense_threshold = thr;
        CK(cudaMemsetAsync(p->d_dense, 0, sizeof(int32_t), s));
        dense_classify_kernel<G><<<blocks(p->n, 8), 256, 0, s>>>(a, cfg);
        CK(cudaGetLastError());
      }
      const int r = patch();
      if (r || thr == INT32_MAX) return r;
      a.env_list = p->d_dense + 8;
      a.env_count = p->d_dense;
      return with_layout(mode, [&](auto m) { return launch_render<G, decltype(m)::value>(a, cfg, smem_total, s); });
    }
  });
}

struct DualRender { const uint32_t *planes2; const uint8_t *reset_flags; int stack_k, stack_slot, stack_mode; };
static int render_impl(tbx_pool *p, uint8_t *dst, int mode, int out_w, int out_h, void *stream, const DualRender *dual) {
  if (!p || !dst) return set_err(TBX_EINVAL, "pool/dst is NULL");
  if (((uintptr_t)dst & 15) != 0) return set_err(TBX_EINVAL, "dst must be 16-byte aligned");
  size_t fb = tbx_obs_bytes(p, mode, out_w, out_h);
  if (fb == 0) return set_err(TBX_EINVAL, "unsupported observation layout or size");
  CK(cudaSetDevice(p->device));
  int r = ensure_base(p);
  if (r) return r;
  const int pix = obs_pix(mode);
  RenderArgs a = {};
  a.planes = p->planes; a.n = p->n; a.n_pad = p->n_pad; a.cfg = p->d_cfg; a.tables = p->d_tables;
  a.planes2 = dual ? dual->planes2 : 0; a.reset_flags = dual ? dual->reset_flags : 0;
  a.stack_k = dual ? dual->stack_k : 1; a.stack_slot = dual ? dual->stack_slot : 0; a.stack_mode = dual ? dual->stack_mode : 0; a.env_stride = fb * (size_t)a.stack_k;
  a.dst = dst; a.frame_bytes = fb;
  for (int b = 0; b < 2; b++) a.base[b] = pix == 4 ? p->base->rgba[b] : pix == 3 ? p->base->rgb[b] : p->base->gray[b];
  a.smem_canvas = align16(p->info->rec_words * TBX_EPC * 4) * (dual ? 2 : 1);
  cudaStream_t s = (cudaStream_t)stream;
  if (mode == TBX_OBS_GRAY_AREA || mode == TBX_OBS_RGB_AREA) return render_area(p, a, out_w, out_h, mode == TBX_OBS_RGB_AREA, s);
  return render_native(p, a, mode, s);
}

extern "C" {

int tbx_render(tbx_pool *p, uint8_t *dst, int mode, int out_w, int out_h, void *stream) {
  return guarded([&] { return render_impl(p, dst, mode, out_w, out_h, stream, 0); });
}

} /* extern "C" */

/* ---- the fused wrapper stack (tbx_wrap.cuh) */
struct tbx_wrap {
  tbx_pool *pool;
  int skip, noop_max, episodic_life, fire_reset, clip_rewards, stack_k, out_w, out_h;
  uint64_t noop_seed, env0;
  Buf<uint32_t> planes_prev, wstate;
  Buf<uint8_t> was_reset;
  int head; /* ring slot of the newest frame */
  int stack_mode; /* what a reset observation does to the other k-1 ring slots: 0 = fills them (FrameStack.reset), 1 = zeroes them (VecFrameStack) */
  int obs_mode;   /* the ring's layout: TBX_OBS_GRAY_AREA or TBX_OBS_RGB_AREA (WarpFrame(grayscale=False)) */
  bool stepped;   /* tbx_wrap_step has run: the ring holds frames of obs_mode's layout */
  int32_t *ep_return, *ep_length; /* caller-owned device outputs of Monitor's episode record, or NULL */
  int words;               /* wrapper words per env in wstate: 5, or 7 with sticky actions (tbx_wrap.cuh) */
  uint64_t sticky_seed, sticky_thr; /* sticky actions: the draw's seed and llround(p * 2^32); thr 0 = off */
  int max_steps;           /* episode time limit in agent steps, 0 = none */
  uint8_t *truncated;      /* caller-owned device output, or NULL */
};
static const int TBX_WRAP_WORDS_MAX = 7; /* wstate is allocated for the sticky layout */

extern "C" {

int tbx_wrap_create(tbx_pool *p, int skip, int noop_max, int episodic_life, int fire_reset, int clip_rewards, int stack_k, int out_w, int out_h,
                    uint64_t noop_seed, uint64_t env0, tbx_wrap **out) {
  if (!p || !out) return set_err(TBX_EINVAL, "pool/out is NULL");
  *out = 0;
  if (skip < 1 || skip > 64 || noop_max < 0 || noop_max > 1000 || stack_k < 1 || stack_k > 16) return set_err(TBX_EINVAL, "skip / noop_max / stack_k out of range");
  if (tbx_obs_bytes(p, TBX_OBS_GRAY_AREA, out_w, out_h) == 0) return set_err(TBX_EINVAL, "unsupported observation size");
  CK(cudaSetDevice(p->device));
  return guarded([&]() -> int {
    std::unique_ptr<tbx_wrap> w(new tbx_wrap());
    w->pool = p; w->skip = skip; w->noop_max = noop_max; w->episodic_life = episodic_life; w->fire_reset = fire_reset; w->clip_rewards = clip_rewards;
    w->stack_k = stack_k; w->out_w = out_w; w->out_h = out_h; w->noop_seed = noop_seed; w->env0 = env0; w->obs_mode = TBX_OBS_GRAY_AREA;
    const size_t plane_words = (size_t)p->info->rec_words * p->n_pad;
    cudaError_t e = w->planes_prev.alloc(plane_words);
    w->words = 5;
    if (e == cudaSuccess) e = w->wstate.alloc(TBX_WRAP_WORDS_MAX * (size_t)p->n_pad);
    if (e == cudaSuccess) e = w->was_reset.alloc((size_t)p->n_pad);
    if (e == cudaSuccess) e = cudaMemcpy(w->planes_prev, p->planes, plane_words * 4, cudaMemcpyDeviceToDevice);
    if (e == cudaSuccess) e = cudaMemset(w->wstate, 0, TBX_WRAP_WORDS_MAX * (size_t)p->n_pad * 4);
    if (e == cudaSuccess) { /* EpisodicLifeEnv.__init__: lives = 0, was_real_done = True (atari_wrappers.py:155-156) */
      std::vector<uint32_t> ones((size_t)p->n_pad, 1u);
      e = cudaMemcpy(w->wstate + p->n_pad, ones.data(), ones.size() * 4, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMemset(w->was_reset, 0, (size_t)p->n_pad);
    if (e != cudaSuccess) return set_err(TBX_ECUDA, std::string("tbx_wrap_create: ") + cudaGetErrorString(e));
    *out = w.release();
    return TBX_OK;
  });
}

int tbx_wrap_set_stack_mode(tbx_wrap *w, int mode) {
  if (!w || (mode != 0 && mode != 1)) return set_err(TBX_EINVAL, "wrap is NULL or unknown stack mode (0 = FrameStack, 1 = VecFrameStack)");
  w->stack_mode = mode;
  return TBX_OK;
}
int tbx_wrap_set_obs_mode(tbx_wrap *w, int obs_mode) {
  if (!w || (obs_mode != TBX_OBS_GRAY_AREA && obs_mode != TBX_OBS_RGB_AREA))
    return set_err(TBX_EINVAL, "wrap is NULL or unsupported observation layout (TBX_OBS_GRAY_AREA or TBX_OBS_RGB_AREA)");
  if (w->stepped) return set_err(TBX_EINVAL, "the observation layout is set before the first tbx_wrap_step");
  w->obs_mode = obs_mode;
  return TBX_OK;
}
int tbx_wrap_set_sticky_actions(tbx_wrap *w, double repeat_action_probability, uint64_t seed) {
  const double p = repeat_action_probability;
  if (!w || !(p >= 0.0 && p <= 1.0)) return set_err(TBX_EINVAL, "wrap is NULL or repeat_action_probability is not in [0, 1]");
  if (w->stepped) return set_err(TBX_EINVAL, "sticky actions are set before the first tbx_wrap_step");
  const int words = p > 0.0 ? 7 : 5;
  if (words == 7) { /* the remembered ALE id (NOOP) and the frame counter of every env start at 0 */
    CK(cudaSetDevice(w->pool->device));
    CK(cudaMemset(w->wstate + 5 * (size_t)w->pool->n_pad, 0, 2 * (size_t)w->pool->n_pad * 4));
  }
  w->words = words;
  w->sticky_seed = seed;
  w->sticky_thr = (uint64_t)llround(p * 4294967296.0);
  return TBX_OK;
}
int tbx_wrap_set_time_limit(tbx_wrap *w, int max_episode_steps, uint8_t *truncated_dev) {
  if (!w || max_episode_steps < 0) return set_err(TBX_EINVAL, "wrap is NULL or max_episode_steps < 0");
  if (w->stepped) return set_err(TBX_EINVAL, "the time limit is set before the first tbx_wrap_step");
  w->max_steps = max_episode_steps;
  w->truncated = truncated_dev;
  return TBX_OK;
}
int tbx_wrap_set_episode_outputs(tbx_wrap *w, int32_t *ep_return_dev, int32_t *ep_length_dev) {
  if (!w) return set_err(TBX_EINVAL, "wrap is NULL");
  w->ep_return = ep_return_dev; w->ep_length = ep_length_dev;
  return TBX_OK;
}

int tbx_wrap_destroy(tbx_wrap *w) {
  if (!w) return TBX_OK;
  cudaSetDevice(w->pool->device);
  cudaDeviceSynchronize();
  delete w;
  return TBX_OK;
}

int tbx_wrap_step(tbx_wrap *w, const int32_t *actions, uint8_t *obs_ring, int32_t *reward, uint8_t *done, uint8_t *real_done, int32_t *score,
                  int32_t *lives, int *slot_out, void *stream) {
  if (!w) return set_err(TBX_EINVAL, "wrap is NULL");
  tbx_pool *p = w->pool;
  CK(cudaSetDevice(p->device));
  cudaStream_t s = (cudaStream_t)stream;
  w->stepped = true;
  WrapArgs a;
  a.planes = p->planes; a.planes_prev = w->planes_prev; a.wstate = w->wstate; a.n = p->n; a.n_pad = p->n_pad; a.cfg = p->d_cfg; a.tables = p->d_tables;
  a.legal = p->d_legal; a.n_legal = p->info->n_legal; a.actions = actions;
  a.skip = w->skip; a.noop_max = w->noop_max; a.episodic_life = w->episodic_life; a.fire_reset = w->fire_reset; a.clip_rewards = w->clip_rewards;
  a.noop_seed = w->noop_seed; a.env0 = w->env0;
  a.reward = reward; a.score = score; a.lives = lives; a.done = done; a.real_done = real_done; a.was_reset = w->was_reset;
  a.ep_return = w->ep_return; a.ep_length = w->ep_length;
  a.sticky_seed = w->sticky_seed; a.sticky_thr = w->sticky_thr; a.max_steps = w->max_steps; a.truncated = w->truncated;
  a.stats = p->d_stats; a.bad_actions = p->d_bad;
  with_game(p->game, [&](auto g) {
    constexpr int G = decltype(g)::value;
    if (w->words == 7) wrap_step_kernel<G, true><<<blocks(p->n, 128), 128, 0, s>>>(a);
    else wrap_step_kernel<G, false><<<blocks(p->n, 128), 128, 0, s>>>(a);
  });
  CK(cudaGetLastError());
  if (obs_ring) {
    w->head = (w->head + 1) % w->stack_k;
    DualRender d;
    d.planes2 = w->planes_prev; d.reset_flags = w->was_reset; d.stack_k = w->stack_k; d.stack_slot = w->head; d.stack_mode = w->stack_mode;
    int r = guarded([&] { return render_impl(p, obs_ring, w->obs_mode, w->out_w, w->out_h, stream, &d); });
    if (r) return r;
  }
  if (slot_out) *slot_out = w->head;
  return TBX_OK;
}

int tbx_field_lookup(const char *game, const char *path, int *word, int *kind, int *bit) {
  int g = tbx::game_from_name(game);
  if (g < 0 || !path) return set_err(TBX_EINVAL, "unknown game or NULL path");
  tbxfields::Field f;
  if (!tbxfields::lookup(g, path, &f)) return set_err(TBX_EINVAL, std::string("no scalar state property '") + path + "' for " + game);
  if (word) *word = f.word;
  if (kind) *kind = f.kind;
  if (bit) *bit = f.bit;
  return TBX_OK;
}
static int field_of(tbx_pool *p, const char *path, tbxfields::Field *f) {
  if (!p || !path) return set_err(TBX_EINVAL, "pool/path is NULL");
  if (!tbxfields::lookup(p->game, path, f)) return set_err(TBX_EINVAL, std::string("no scalar state property '") + path + "' for " + p->info->name);
  return TBX_OK;
}
int tbx_field_get(tbx_pool *p, const char *path, void *out, void *stream) {
  tbxfields::Field f;
  int r = field_of(p, path, &f);
  if (r) return r;
  if (!out) return set_err(TBX_EINVAL, "out is NULL");
  CK(cudaSetDevice(p->device));
  field_get_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(p->planes, p->n, p->n_pad, f.word, f.kind, f.bit < 0 ? 0 : f.bit,
                                                                         (int32_t *)out, (double *)out);
  CK(cudaGetLastError());
  return TBX_OK;
}
int tbx_field_set(tbx_pool *p, const char *path, const void *values, const uint8_t *mask, void *stream) {
  tbxfields::Field f;
  int r = field_of(p, path, &f);
  if (r) return r;
  if (!values) return set_err(TBX_EINVAL, "values is NULL");
  CK(cudaSetDevice(p->device));
  const int also = (f.kind == TBX_F_I32 && f.word == TBX_FW(TbxHdr, score)) ? TBX_FW(TbxHdr, prev_score) : -1;
  field_set_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(p->planes, p->n, p->n_pad, f.word, f.kind, f.bit < 0 ? 0 : f.bit,
                                                                         (const int32_t *)values, (const double *)values, mask, also);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_breakout_columns(tbx_pool *p, int op, int col, const uint8_t *mask, int32_t *out, void *stream) {
  if (!p || p->game != TBX_BREAKOUT) return set_err(TBX_EINVAL, "tbx_breakout_columns needs a breakout pool");
  if (op < 0 || op > 2 || (op == 2 && !out)) return set_err(TBX_EINVAL, "op is 0 (remove column), 1 (fill column) or 2 (count channels into out)");
  CK(cudaSetDevice(p->device));
  brk_column_kernel<<<blocks(p->n, 128), 128, 0, (cudaStream_t)stream>>>(p->planes, p->n, p->n_pad, reinterpret_cast<const BrkTable *>(p->d_tables.get()), op, col, mask, out);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_read_scalars(tbx_pool *p, int32_t *score, int32_t *lives, int32_t *level, void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  CK(cudaSetDevice(p->device));
  read_scalars_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(p->planes, p->n, p->n_pad, score, lives, level);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_fill_actions(tbx_pool *p, int32_t *actions, uint64_t seed, uint64_t env0, uint64_t t, void *stream) {
  if (!p || !actions) return set_err(TBX_EINVAL, "pool/actions is NULL");
  CK(cudaSetDevice(p->device));
  fill_actions_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(actions, p->n, seed, env0, t, p->d_legal, p->info->n_legal);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_fill_actions_at(tbx_pool *p, int32_t *actions, uint64_t seed, uint64_t env0, const uint64_t *t_dev, void *stream) {
  if (!p || !actions || !t_dev) return set_err(TBX_EINVAL, "pool/actions/t_dev is NULL");
  CK(cudaSetDevice(p->device));
  fill_actions_at_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(actions, p->n, seed, env0, t_dev, p->d_legal, p->info->n_legal);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_fill_actions_policy(tbx_pool *p, int32_t *actions, int policy, uint64_t t, void *stream) {
  if (!p || !actions) return set_err(TBX_EINVAL, "pool/actions is NULL");
  if (policy != 1 || p->game != TBX_BREAKOUT) return set_err(TBX_EINVAL, "only policy 1 (Breakout ball tracking) is implemented");
  CK(cudaSetDevice(p->device));
  breakout_tracking_actions_kernel<<<blocks(p->n, 256), 256, 0, (cudaStream_t)stream>>>(p->planes, p->n, p->n_pad, actions, t);
  CK(cudaGetLastError());
  return TBX_OK;
}

int tbx_stats_read(tbx_pool *p, int64_t *out, int reset, void *stream) {
  if (!p || !out) return set_err(TBX_EINVAL, "pool/out is NULL");
  CK(cudaSetDevice(p->device));
  cudaStream_t s = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(out, p->d_stats, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (reset) CK(cudaMemsetAsync(p->d_stats, 0, 4 * sizeof(int64_t), s));
  return TBX_OK;
}

int tbx_stats_read_device(tbx_pool *p, int64_t *out_dev, void *stream) {
  if (!p || !out_dev) return set_err(TBX_EINVAL, "pool/out is NULL");
  CK(cudaSetDevice(p->device));
  CK(cudaMemcpyAsync(out_dev, p->d_stats, 4 * sizeof(int64_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return TBX_OK;
}

int tbx_step_host(tbx_pool *p, const int32_t *actions, int auto_reset, int mode, int out_w, int out_h, uint8_t *obs, int32_t *reward,
                  uint8_t *done, int32_t *score, int32_t *lives) {
  if (!p || !actions) return set_err(TBX_EINVAL, "pool/actions is NULL");
  CK(cudaSetDevice(p->device));
  const size_t n = (size_t)p->n;
  return guarded([&]() -> int {
    if (!p->hs) {
      auto h = std::make_unique<HostStaging>();
      CK(cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking));
      CK(h->actions.alloc(n)); CK(h->reward.alloc(n)); CK(h->score.alloc(n)); CK(h->lives.alloc(n)); CK(h->done.alloc(n));
      p->hs = std::move(h);
    }
    HostStaging &h = *p->hs;
    size_t fb = 0;
    if (obs) {
      fb = tbx_obs_bytes(p, mode, out_w, out_h);
      if (fb == 0) return set_err(TBX_EINVAL, "unsupported observation layout or size");
      if (h.obs.size() < fb * n) CK(cudaStreamSynchronize(h.s));
      CK(h.obs.grow(fb * n));
    }
    CK(cudaMemcpyAsync(h.actions, actions, n * 4, cudaMemcpyHostToDevice, h.s));
    int r = do_step(p, h.actions, 0, auto_reset, h.reward, h.done, h.score, h.lives, h.s);
    if (r) return r;
    if (reward) CK(cudaMemcpyAsync(reward, h.reward, n * 4, cudaMemcpyDeviceToHost, h.s));
    if (done) CK(cudaMemcpyAsync(done, h.done, n, cudaMemcpyDeviceToHost, h.s));
    if (score) CK(cudaMemcpyAsync(score, h.score, n * 4, cudaMemcpyDeviceToHost, h.s));
    if (lives) CK(cudaMemcpyAsync(lives, h.lives, n * 4, cudaMemcpyDeviceToHost, h.s));
    if (obs) {
      r = render_impl(p, h.obs, mode, out_w, out_h, h.s, 0);
      if (r) return r;
      CK(cudaMemcpyAsync(obs, h.obs, fb * n, cudaMemcpyDeviceToHost, h.s));
    }
    CK(cudaStreamSynchronize(h.s));
    int bad = 0;
    CK(cudaMemcpy(&bad, p->d_bad, sizeof bad, cudaMemcpyDeviceToHost));
    if (bad) { cudaMemset(p->d_bad, 0, sizeof(int)); return set_err(TBX_EACTION, "Expected to apply action, but failed: invalid ALE action id"); }
    return TBX_OK;
  });
}

/* ---- JSON */
static char *dup_str(const std::string &s) {
  char *out = (char *)malloc(s.size() + 1);
  if (out) memcpy(out, s.c_str(), s.size() + 1);
  return out;
}
void tbx_free_str(char *s) { free(s); }

static int ensure_json_staging(tbx_pool *p, int n) {
  const size_t words = (size_t)n * p->info->rec_words;
  CK(p->j_ids.grow(n, std::max<size_t>(1024, (size_t)n * 2)));
  const size_t cap = std::max<size_t>((size_t)1024 * p->info->rec_words, words * 2);
  CK(p->j_recs.grow(words, cap));
  CK(p->j_host.grow(words, cap));
  return TBX_OK;
}
/* records of the listed envs -> p->j_host (AoS).  Runs on the legacy default stream, which is ordered after the work of
 * every blocking stream; callers on non-blocking streams synchronise first (the Python layer does). */
static int fetch_records(tbx_pool *p, const int32_t *ids, int n) {
  const int rw = p->info->rec_words;
  for (int i = 0; i < n; i++) if (ids[i] < 0 || ids[i] >= p->n) return set_err(TBX_EINVAL, "env id out of range");
  CK(cudaSetDevice(p->device));
  int r = ensure_json_staging(p, n);
  if (r) return r;
  if (p->hs) CK(cudaStreamSynchronize(p->hs->s));
  CK(cudaMemcpyAsync(p->j_ids, ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, 0));
  gather_kernel<<<blocks(n * rw, 256), 256>>>(p->planes, p->n_pad, p->j_ids, n, rw, p->j_recs);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(p->j_host, p->j_recs, (size_t)n * rw * 4, cudaMemcpyDeviceToHost, 0));
  CK(cudaStreamSynchronize(0));
  return TBX_OK;
}
/* p->j_host (AoS) -> the listed envs; the ids are still on the device from fetch_records */
static int store_records(tbx_pool *p, int n) {
  const int rw = p->info->rec_words;
  CK(cudaMemcpyAsync(p->j_recs, p->j_host, (size_t)n * rw * 4, cudaMemcpyHostToDevice, 0));
  scatter_kernel<<<blocks(n * rw, 256), 256>>>(p->planes, p->n_pad, p->j_ids, n, rw, p->j_recs);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(0));
  return TBX_OK;
}

int tbx_state_to_json(tbx_pool *p, const int32_t *ids, int n, char **out) {
  if (!p || !ids || !out || n < 0) return set_err(TBX_EINVAL, "bad arguments");
  for (int i = 0; i < n; i++) out[i] = 0;
  if (n == 0) return TBX_OK;
  const int r = guarded([&]() -> int {
    int r = fetch_records(p, ids, n);
    if (r) return r;
    const int rw = p->info->rec_words;
    const uint32_t *recs = p->j_host;
    with_game(p->game, [&](auto g) {
      constexpr int G = decltype(g)::value;
      const auto &tabs = tables<G>(p);
      parallel_for(n, [&](int i) {
        const auto &rec = *reinterpret_cast<const typename Traits<G>::Rec *>(recs + (size_t)i * rw);
        const typename Traits<G>::Table *t = 0;
        if constexpr (kTables<G>) {
          if (rec.hdr.tbl < 0 || rec.hdr.tbl >= (int)tabs.size()) throw std::runtime_error("corrupt table index");
          t = &tabs[rec.hdr.tbl];
        }
        out[i] = dup_str(tbxjson::dump(state_to_json(rec, t)));
        if (!out[i]) throw std::runtime_error("out of host memory");
      });
    });
    return TBX_OK;
  });
  if (r) for (int i = 0; i < n; i++) { free(out[i]); out[i] = 0; }
  return r;
}

int tbx_state_from_json(tbx_pool *p, const int32_t *ids, int n, const char *const *json) {
  if (!p || !ids || !json || n < 0) return set_err(TBX_EINVAL, "bad arguments");
  if (n == 0) return TBX_OK;
  return guarded([&]() -> int {
    int r = fetch_records(p, ids, n); /* keeps the fields JSON does not carry (simulator rand, episode counters) */
    if (r) return r;
    const int rw = p->info->rec_words;
    uint32_t *recs = p->j_host;
    with_game(p->game, [&](auto g) {
      constexpr int G = decltype(g)::value;
      typedef typename Traits<G>::Rec Rec;
      /* parse everything (in parallel) before touching the pool so a bad document leaves it unchanged */
      Tables<G> new_tabs(kTables<G> ? n : 0);
      parallel_for(n, [&](int i) {
        Rec &rec = *reinterpret_cast<Rec *>(recs + (size_t)i * rw);
        const Value v = tbxjson::parse(json[i]);
        if constexpr (kTables<G>) { state_from_json(v, rec, new_tabs[i]); fit_table(p->cfg, new_tabs[i]); }
        else tbx::si_state_from_json(v, rec);
      });
      for (int i = 0; i < (int)new_tabs.size(); i++) reinterpret_cast<Rec *>(recs + (size_t)i * rw)->hdr.tbl = intern(tables<G>(p), new_tabs[i]);
    });
    r = upload_tables(p);
    if (r) return r;
    return store_records(p, n);
  });
}

int tbx_config_to_json(tbx_pool *p, char **out) {
  if (!p || !out) return set_err(TBX_EINVAL, "bad arguments");
  /* ctoybox's config_to_json shows the simulator as it is NOW: `rand` is the simulator rng that new_game has advanced.
   * A pool keeps one simulator rng per env; the pool-level document reports env 0's (the batch-1 shim's only env). */
  tbx::Config c = p->cfg;
  CK(cudaSetDevice(p->device));
  uint32_t w[4];
  CK(cudaMemcpy2D(w, sizeof(uint32_t), p->planes + (size_t)TBX_HW(sim_rand) * p->n_pad, (size_t)p->n_pad * sizeof(uint32_t), sizeof(uint32_t), 4,
                  cudaMemcpyDeviceToHost));
  cfg_rand(c)[0] = (uint64_t)w[0] | ((uint64_t)w[1] << 32);
  cfg_rand(c)[1] = (uint64_t)w[2] | ((uint64_t)w[3] << 32);
  return guarded([&] {
    *out = dup_str(tbxjson::dump(tbx::config_to_json(c)));
    return *out ? TBX_OK : set_err(TBX_ENOMEM, "out of host memory");
  });
}
int tbx_config_from_json(tbx_pool *p, const char *json) {
  if (!p || !json) return set_err(TBX_EINVAL, "bad arguments");
  return guarded([&]() -> int {
    tbx::Config c = p->cfg;
    tbx::config_from_json(c, tbxjson::parse(json));
    CK(cudaSetDevice(p->device));
    CK(cudaDeviceSynchronize());
    p->cfg = c;
    drop_render_cache(p);
    install_default_table(p);
    int r = upload_tables(p);
    if (r) return r;
    /* write_config_json replaces the simulator, its rng included: every env's simulator rng restarts from the document's */
    set_sim_rand_kernel<<<blocks(p->n, 256), 256>>>(p->planes, p->n, p->n_pad, cfg_rand(p->cfg)[0], cfg_rand(p->cfg)[1]);
    CK(cudaGetLastError());
    return upload_cfg(p);
  });
}
int tbx_schema_for_state(const char *game, char **out) {
  int g = tbx::game_from_name(game);
  if (g < 0 || !out) return set_err(TBX_EINVAL, "unknown game");
  return guarded([&] {
    *out = dup_str(tbxjson::dump(tbx::schema_for_state(g)));
    return *out ? TBX_OK : set_err(TBX_ENOMEM, "out of host memory");
  });
}
int tbx_schema_for_config(const char *game, char **out) {
  int g = tbx::game_from_name(game);
  if (g < 0 || !out) return set_err(TBX_EINVAL, "unknown game");
  return guarded([&] {
    *out = dup_str(tbxjson::dump(tbx::schema_for_config(g)));
    return *out ? TBX_OK : set_err(TBX_ENOMEM, "out of host memory");
  });
}
int tbx_query_json(tbx_pool *p, int env, const char *query, const char *args_json, char **out) {
  if (!p || !query || !out) return set_err(TBX_EINVAL, "bad arguments");
  *out = 0;
  if (env < 0 || env >= p->n) return set_err(TBX_EINVAL, "env id out of range");
  return guarded([&]() -> int {
    Value args = tbxjson::parse(args_json ? args_json : "null");
    std::string q(query);
    const uint32_t *rec = 0;
    const BrkTable *brk = 0;
    if (p->game == TBX_BREAKOUT) {
      int32_t id = env;
      int r = fetch_records(p, &id, 1);
      if (r) return r;
      rec = p->j_host;
      int tbl = reinterpret_cast<const BrkRec *>(rec)->hdr.tbl;
      if (tbl < 0 || tbl >= (int)tables<TBX_BREAKOUT>(p).size()) return set_err(TBX_EINVAL, "corrupt table index");
      brk = &tables<TBX_BREAKOUT>(p)[tbl];
    }
    Value res = tbx::query_json(p->game, rec, brk, q, args);
    *out = dup_str(tbxjson::dump(res));
    return *out ? TBX_OK : set_err(TBX_ENOMEM, "out of host memory");
  });
}

} /* extern "C" */

/* ---- device-resident state snapshots (tbx_snapshot.cuh) */
/* the pool's interned tables as bytes */
struct TableView { const void *data; size_t bytes; int count; };
static TableView table_view(const tbx_pool *p) {
  return with_game(p->game, [&](auto g) {
    constexpr int G = decltype(g)::value;
    const auto &t = tables<G>(p);
    return TableView{t.data(), kTables<G> ? sizeof t[0] : 0, (int)t.size()};
  });
}

static int state_tables(const tbx_pool *p, int rows, void *out, size_t cap, size_t *size) {
  const TableView t = table_view(p);
  const tbx_state_blob_header h = {TBX_STATE_MAGIC, TBX_STATE_FORMAT, (uint32_t)p->game, (uint32_t)rows, (uint32_t)t.bytes, (uint32_t)t.count};
  const size_t need = sizeof h + (size_t)h.table_bytes * h.table_count;
  *size = need;
  if (!out) return TBX_OK;
  if (cap < need) return set_err(TBX_EINVAL, "the tables blob needs " + std::to_string(need) + " bytes, the buffer holds " + std::to_string(cap));
  memcpy(out, &h, sizeof h);
  if (need > sizeof h) memcpy((char *)out + sizeof h, t.data, need - sizeof h);
  return TBX_OK;
}
/* the pool side of a copy: planes, then (wrapped env) its `words` wrapper words */
static SnapSide pool_side(const tbx_pool *p, uint32_t *wstate, const int32_t *ids) {
  SnapSide s;
  s.base0 = p->planes; s.split = p->info->rec_words; s.stride = (size_t)p->n_pad;
  s.base1 = wstate ? wstate : p->planes + (size_t)s.split * p->n_pad;
  s.idx = ids; s.lim = p->n;
  return s;
}
static SnapSide snap_side(uint32_t *snap, int k, int rows, const int32_t *cols) {
  SnapSide s;
  s.base0 = snap; s.split = rows; s.stride = (size_t)k; s.base1 = snap + (size_t)rows * k;
  s.idx = cols; s.lim = k;
  return s;
}
static int launch_snap_copy(const SnapArgs &a, cudaStream_t s) {
  if (a.owner) {
    snap_owner_kernel<<<blocks(a.k, TBX_SNAP_THREADS), TBX_SNAP_THREADS, 0, s>>>(a);
    CK(cudaGetLastError());
  }
  snap_copy_kernel<<<dim3(blocks(a.k, TBX_SNAP_THREADS), blocks(a.rows, TBX_SNAP_ROWS)), TBX_SNAP_THREADS, 0, s>>>(a);
  CK(cudaGetLastError());
  return TBX_OK;
}

static int state_save(tbx_pool *p, uint32_t *wstate, int words, const int32_t *ids, int k, uint32_t *snap, cudaStream_t s) {
  if (!snap || k < 0) return set_err(TBX_EINVAL, "snap is NULL or k < 0");
  if (!ids && k > p->n) return set_err(TBX_EINVAL, "without env ids, k must not exceed the pool's env count");
  if (k == 0) return TBX_OK;
  CK(cudaSetDevice(p->device));
  SnapArgs a;
  a.rows = p->info->rec_words + (wstate ? words : 0);
  a.src = pool_side(p, wstate, ids); a.dst = snap_side(snap, k, a.rows, 0);
  a.k = k; a.tbl_row = -1; a.tbl_lim = -1; a.remap = 0; a.owner = 0; a.bad = p->d_bad + 1;
  return launch_snap_copy(a, s);
}

/* The tables a snapshot was saved with.  Byte-identical to the pool's first `count` tables (the pool's own snapshots, and
 * those of pools with the same config): *remap = NULL and tbl is copied as is, a host-only check.  Otherwise every blob table
 * is interned into this pool (delta_ok recomputed for this pool's config first, as tbx_state_from_json does) and *remap maps
 * blob indices to pool indices; that path synchronises the device. */
static int snapshot_remap(tbx_pool *p, const uint8_t *tabs, int count, const int32_t **remap) {
  *remap = 0;
  std::vector<int32_t> map;
  bool identity = true;
  with_game(p->game, [&](auto g) {
    constexpr int G = decltype(g)::value;
    if constexpr (kTables<G>) {
      auto &v = tables<G>(p);
      typename Traits<G>::Table t;
      if (count <= (int)v.size() && memcmp(tabs, v.data(), (size_t)count * sizeof t) == 0) return;
      for (int i = 0; i < count; i++) {
        memcpy(&t, tabs + (size_t)i * sizeof t, sizeof t);
        fit_table(p->cfg, t);
        map.push_back(intern(v, t));
        identity = identity && map[i] == i;
      }
    }
  });
  if (map.empty()) return TBX_OK;
  int r = upload_tables(p);
  if (r) return r;
  if (identity) return TBX_OK;
  CK(cudaDeviceSynchronize()); /* an earlier load may still read the remap buffer */
  CK(p->d_remap.grow(count));
  CK(cudaMemcpy(p->d_remap, map.data(), (size_t)count * sizeof(int32_t), cudaMemcpyHostToDevice));
  *remap = p->d_remap;
  return TBX_OK;
}
static int state_load(tbx_pool *p, uint32_t *wstate, int words, const uint32_t *snap, int k_snap, const int32_t *cols, const int32_t *ids, int n, const void *blob,
                      size_t blob_bytes, cudaStream_t s) {
  const int rows = p->info->rec_words + (wstate ? words : 0);
  if (k_snap < 0 || n < 0 || (n > 0 && !snap)) return set_err(TBX_EINVAL, "snap is NULL, or k_snap / n < 0");
  tbx_state_blob_header h;
  if (!blob || blob_bytes < sizeof h) return set_err(TBX_EINVAL, "state snapshot: the tables blob is missing or truncated");
  memcpy(&h, blob, sizeof h);
  if (h.magic != TBX_STATE_MAGIC) return set_err(TBX_EINVAL, "state snapshot: not a tables blob (bad magic)");
  if (h.format != TBX_STATE_FORMAT)
    return set_err(TBX_EINVAL, "state snapshot: format " + std::to_string(h.format) + ", this library reads format " + std::to_string(TBX_STATE_FORMAT));
  if (h.game != (uint32_t)p->game) return set_err(TBX_EINVAL, std::string("state snapshot: saved from another game, this pool runs ") + p->info->name);
  if (h.rows != (uint32_t)rows)
    return set_err(TBX_EINVAL, "state snapshot: " + std::to_string(h.rows) + " rows per env, this " + (wstate ? "wrapped env" : "pool") + " needs " + std::to_string(rows));
  if (h.table_bytes != table_view(p).bytes || h.table_count > (1u << 20) || blob_bytes != sizeof h + (size_t)h.table_bytes * h.table_count)
    return set_err(TBX_EINVAL, "state snapshot: the tables blob's size does not match its header");
  if (n == 0) return TBX_OK;
  CK(cudaSetDevice(p->device));
  const int32_t *remap = 0;
  int r = snapshot_remap(p, (const uint8_t *)blob + sizeof h, (int)h.table_count, &remap);
  if (r) return r;
  if (ids) CK(p->d_owner.grow(p->n_pad));
  SnapArgs a;
  a.rows = rows;
  a.src = snap_side(const_cast<uint32_t *>(snap), k_snap, rows, cols); a.dst = pool_side(p, wstate, ids);
  a.k = n; a.tbl_row = p->game == TBX_SPACE_INVADERS ? -1 : TBX_HW(tbl); a.tbl_lim = (int)h.table_count; a.remap = remap;
  a.owner = ids ? p->d_owner.get() : 0; a.bad = p->d_bad + 1;
  if (a.owner) CK(cudaMemsetAsync(p->d_owner, 0xff, (size_t)p->n_pad * sizeof(int32_t), s)); /* -1: no entry yet */
  return launch_snap_copy(a, s);
}

extern "C" {

int tbx_state_rows(const tbx_pool *p) { return p ? p->info->rec_words : 0; }
int tbx_wrap_state_rows(const tbx_wrap *w) { return w ? w->pool->info->rec_words + w->words : 0; }
int tbx_state_tables(const tbx_pool *p, void *out_host, size_t cap, size_t *size) {
  if (!p || !size) return set_err(TBX_EINVAL, "pool/size is NULL");
  return state_tables(p, p->info->rec_words, out_host, cap, size);
}
int tbx_wrap_state_tables(const tbx_wrap *w, void *out_host, size_t cap, size_t *size) {
  if (!w || !size) return set_err(TBX_EINVAL, "wrap/size is NULL");
  return state_tables(w->pool, w->pool->info->rec_words + w->words, out_host, cap, size);
}
int tbx_state_save(tbx_pool *p, const int32_t *ids_dev, int k, uint32_t *snap_dev, void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  return state_save(p, 0, 0, ids_dev, k, snap_dev, (cudaStream_t)stream);
}
int tbx_wrap_state_save(tbx_wrap *w, const int32_t *ids_dev, int k, uint32_t *snap_dev, void *stream) {
  if (!w) return set_err(TBX_EINVAL, "wrap is NULL");
  return state_save(w->pool, w->wstate, w->words, ids_dev, k, snap_dev, (cudaStream_t)stream);
}
int tbx_state_load(tbx_pool *p, const uint32_t *snap_dev, int k_snap, const int32_t *cols_dev, const int32_t *ids_dev, int n, const void *tables_blob,
                   size_t blob_bytes, void *stream) {
  if (!p) return set_err(TBX_EINVAL, "pool is NULL");
  return guarded([&] { return state_load(p, 0, 0, snap_dev, k_snap, cols_dev, ids_dev, n, tables_blob, blob_bytes, (cudaStream_t)stream); });
}
int tbx_wrap_state_load(tbx_wrap *w, const uint32_t *snap_dev, int k_snap, const int32_t *cols_dev, const int32_t *ids_dev, int n, const void *tables_blob,
                        size_t blob_bytes, void *stream) {
  if (!w) return set_err(TBX_EINVAL, "wrap is NULL");
  return guarded([&] { return state_load(w->pool, w->wstate, w->words, snap_dev, k_snap, cols_dev, ids_dev, n, tables_blob, blob_bytes, (cudaStream_t)stream); });
}

} /* extern "C" */
