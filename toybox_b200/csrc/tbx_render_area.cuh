/* tbx_render_area.cuh -- the INTER_AREA (WarpFrame, e.g. 84x84 gray) render kernel: ONE WARP PER ENV, tile based.
 *
 * The reference produces this observation as get_state() (native gray frame, toybox/envs/atari/base.py:109)
 * followed by cv2.resize(..., INTER_AREA) (baselines/baselines/common/atari_wrappers.py:243).  An output frame is
 * only 7 KB, so a CTA-wide shared canvas with barriers between the phases of every env (tbx_render.cuh, used for
 * the native layouts) leaves most issue slots idle.  Here a warp renders its env alone -- no CTA barrier after
 * the record load -- and never materialises the native frame:
 *   1. the pre-computed down-sample of the env's base frame is copied to the destination (16-byte units);
 *   2. the draw-list entries that differ from the base frame are built once (32 slots per pass, one per lane) and
 *      appended, in draw order, to a per-warp list in shared memory; every entry marks the OUTPUT TILES (16 x 8
 *      output pixels) its pixels feed;
 *   3. for every run of horizontally adjacent marked tiles the warp copies the run's source window of the base
 *      frame (a few source rows) into a small shared-memory scratch canvas, paints the list entries that touch it in draw order (painter's
 *      algorithm, identical result to painting the whole frame), and recomputes the tile's output rows that those
 *      entries feed with cv2's exact f32 tap order; the bytes are patched into the destination frame.
 * If an env has more entries than the list holds, its output rows are processed in 2, 4, ... sweeps, each with the
 * entries clipped to the sweep's source rows; if even one tile row overflows, that row is rendered by re-building
 * the primitives per tile (slow, but always correct).
 * Members of a PARALLEL draw-list group cannot conflict, so inside a tile the small solid ones (bricks, maze tiles)
 * are painted lane-parallel; everything else is painted by the whole warp, one entry at a time, in draw order.
 * The kernel renders every plan the library accepts: it is instantiated for 3..5 x 3..4 taps, and for 8 x 8 taps
 * (single frames only) for the plans with more; surplus taps carry zero weight.
 * RGB mode (RGB = true; single frames, and the dual mode of the wrapped path for 3..5 x 3..4 taps): the list, hit tests,
 * sweeps and per-tile rebuild are colour-blind and shared; each entry also keeps its 24-bit colour, and every run is loaded,
 * painted and resolved once per channel from planar base frames (both windows in dual mode), so the scratch window keeps its
 * gray size.  The output is interleaved RGB, = cv2's 3-channel INTER_AREA (which is the per-channel resize).  In dual mode
 * a slot is "in both frames" only if its colour is the same in both, not just its gray.
 */
#ifndef TBX_RENDER_AREA_CUH
#define TBX_RENDER_AREA_CUH
#include "tbx_render.cuh"

namespace tbxk {

#define TBX_TILE_LCAP 128   /* list entries per warp */
#define TBX_TILE_THREADS 256 /* CTA size: 8 warps */
#define TBX_TILE_HSHIFT 3    /* tiles are 16 x (1 << TBX_TILE_HSHIFT) output pixels */
#define TBX_TILE_MAX_RUN 2   /* a run renders at most this many horizontally adjacent tiles through one scratch window */
#ifndef TBX_AREA_MIN_CTAS
#define TBX_AREA_MIN_CTAS 4
#endif
/* the 8 x 8 instantiation keeps its eight column weights per lane in registers: at 4 CTAs per SM (64 registers) it
 * spills, at 2 it needs ~112 and does not */
#define TBX_TILE_MIN_CTAS(TX, TY) ((TX) > 5 || (TY) > 4 ? 2 : TBX_AREA_MIN_CTAS)
/* dual RGB (two scratch windows, the colour array, a channel loop): it spills at 64 and at 80 registers (4 and 3 CTAs per SM)
 * and needs ~128 (2).  Its shared memory allows 4 CTAs per SM for Breakout 84 x 84 (55.5 KB), 3 for Amidar (75.6 KB) and 2 for
 * Space Invaders (90.9 KB) */
#ifndef TBX_TILE_DUAL_RGB_MIN_CTAS
#define TBX_TILE_DUAL_RGB_MIN_CTAS 2
#endif

/* a warp paints one primitive into the tile scratch canvas: window columns [wx0, wx1) (wx0 a multiple of 4, the
 * scratch's column 0), rows [wy0, wy1); `stride` bytes per scratch row */
__device__ __forceinline__ void paint_tile(uint8_t *tile, int stride, int wx0, int wy0, int wx1, int wy1, int qx, int qy, int qw, int qh,
                                           uint32_t val, uint32_t q3, const uint32_t *rec, int lane) {
  const int x0 = max(qx, wx0), x1 = min(qx + qw, wx1), y0 = max(qy, wy0), y1 = min(qy + qh, wy1);
  const int nw = x1 - x0, nh = y1 - y0;
  if (nw <= 0 || nh <= 0) return;
  const int lg = nw > 16 ? 5 : nw > 8 ? 4 : nw > 4 ? 3 : nw > 2 ? 2 : nw > 1 ? 1 : 0;
  const int cpl = 1 << lg, rpp = 32 >> lg, sub = lane >> lg, cx = lane & (cpl - 1);
  const int bw = (q3 >> 16) & 255;
  uint8_t *org = tile + (y0 - wy0) * stride + (x0 - wx0);
  if (bw == 0) {
    for (int yy = sub; yy < nh; yy += rpp)
      for (int xb = cx; xb < nw; xb += cpl) org[yy * stride + xb] = (uint8_t)val;
  } else {
    const uint32_t off = q3 & 0xffffu;
    const bool state = (off & TBX_PRIM_STATE) != 0; /* sprite rows in the env's record (shared) or in the bank (global) */
    const int o = state ? (int)(off & 0x7fffu) : (int)off;
    const int sx = (q3 >> 24) & 15, sy = q3 >> 28;
    const uint32_t ix = d_inv16[sx], iy = d_inv16[sy];
    for (int yy = sub; yy < nh; yy += rpp) {
      const int py = y0 + yy - qy;
      const int sy_i = sy == 1 ? py : (int)(((uint32_t)py * iy) >> 16);
      const uint32_t bits = state ? rec[o + sy_i] : __ldg(&d_bank[o + sy_i]);
      for (int xb = cx; xb < nw; xb += cpl) {
        const int px = x0 + xb - qx;
        const int sx_i = sx == 1 ? px : (int)(((uint32_t)px * ix) >> 16);
        if ((bits >> (bw - 1 - sx_i)) & 1u) org[yy * stride + xb] = (uint8_t)val;
      }
    }
  }
}

/* list entry (uint4) + extent word:
 *   x: x | y << 16;  y: w | h << 16;  z: gray | group << 8 | flags << 16;  w: sprite off | bw << 16 | scale << 24
 *   extent: dxlo | dxhi << 8 | dylo << 16 | dyhi << 24 = the output columns / rows the (clipped) primitive feeds.
 * flags: ENTRY_PAR = member of a PARALLEL draw-list group (no two members conflict, any paint order is right);
 *        ENTRY_SMALL = solid rectangle of at most 128 pixels (one lane can paint it alone). */
#define TBX_ENTRY_PAR 1u
#define TBX_ENTRY_SMALL 2u
#define TBX_ENTRY_DIGIT 4u /* HUD digit with a pre-resolved patch candidate: z bits 24..29 = digit slot index */
template <int W>
__device__ __forceinline__ bool make_entry(const TbxPrim &p, int g, int gmode, int rA, int rB, int dyA, int dyB, const TbxAreaPlan *__restrict__ plan,
                                           uint4 &e, uint32_t &ext) { /* g: group index | 0x80 for the second state of dual mode */
  Clip c;
  if (!clip_prim<W>(p, rA, rB, c)) return false;
  const int dylo = max((int)__ldg(&plan->ydlo[c.y0]), dyA), dyhi = min((int)__ldg(&plan->ydhi[c.y1 - 1]), dyB - 1);
  if (dylo > dyhi) return false;
  const int dxlo = __ldg(&plan->xdlo[c.x0]), dxhi = __ldg(&plan->xdhi[c.x1 - 1]);
  const uint32_t flags = ((gmode & TBX_GROUP_SERIAL) ? 0u : TBX_ENTRY_PAR) | ((p.bw == 0 && (int)p.w * (int)p.h <= 128) ? TBX_ENTRY_SMALL : 0u);
  e.x = (uint32_t)(uint16_t)p.x | ((uint32_t)(uint16_t)p.y << 16);
  e.y = (uint32_t)(uint16_t)p.w | ((uint32_t)(uint16_t)p.h << 16);
  e.z = tbx_luma(p.color) | ((uint32_t)g << 8) | (flags << 16);
  e.w = (uint32_t)p.off | ((uint32_t)p.bw << 16) | ((uint32_t)p.scale << 24);
  ext = (uint32_t)dxlo | ((uint32_t)dxhi << 8) | ((uint32_t)dylo << 16) | ((uint32_t)dyhi << 24);
  return true;
}
/* tiles (16 x (1 << ths) output pixels) are numbered 8 per tile row: bit (ty & 3) * 8 + tx of word ty >> 2 */
__device__ __forceinline__ void mark_tiles(uint32_t *tmask, uint32_t ext, int ths) {
  const int txlo = (ext & 255u) >> 4, txhi = ((ext >> 8) & 255u) >> 4, tylo = ((ext >> 16) & 255u) >> ths, tyhi = (ext >> 24) >> ths;
  const uint32_t cols = ((2u << (txhi - txlo)) - 1u) << txlo;
  for (int ty = tylo; ty <= tyhi; ty++) atomicOr(&tmask[ty >> 2], cols << ((ty & 3) * 8));
}

/* one lane fills its own small solid rectangle in the tile scratch: 32-bit stores over the aligned middle of a row */
__device__ __forceinline__ void paint_tile_lane(uint8_t *tile, int stride, int wx0, int wy0, int wx1, int wy1, int qx, int qy, int qw, int qh, uint32_t val) {
  const int x0 = max(qx, wx0) - wx0, x1 = min(qx + qw, wx1) - wx0, y0 = max(qy, wy0) - wy0, y1 = min(qy + qh, wy1) - wy0;
  if (x0 >= x1 || y0 >= y1) return;
  const int xa = min((x0 + 3) & ~3, x1), xb = max(x1 & ~3, xa);
  const uint32_t w4 = (val & 255u) * 0x01010101u;
  for (int y = y0; y < y1; y++) {
    uint8_t *row = tile + y * stride;
    for (int x = x0; x < xa; x++) row[x] = (uint8_t)val;
    for (int x = xa; x < xb; x += 4) *reinterpret_cast<uint32_t *>(row + x) = w4;
    for (int x = xb; x < x1; x++) row[x] = (uint8_t)val;
  }
}

/* copy the source window [wx0,wx1) x [wy0,wy1) of the base frame into the scratch (wx0, wx1 multiples of 4) */
template <int W>
__device__ __forceinline__ void tile_load(uint8_t *tile, int stride, const uint8_t *bfr, int wx0, int wy0, int wx1, int wy1, int lane) {
  const int nwr = (wx1 - wx0) >> 2, nrows = wy1 - wy0;
  const int lg = nwr > 16 ? 5 : nwr > 8 ? 4 : nwr > 4 ? 3 : 2;
  const int rstep = 32 >> lg;
  for (int cc = lane & ((1 << lg) - 1); cc < nwr; cc += 32) { /* one trip unless the window is wider than 128 bytes */
    const uint32_t *src = reinterpret_cast<const uint32_t *>(bfr + (size_t)wy0 * W + wx0) + cc + (lane >> lg) * (W >> 2);
    uint32_t *dst = reinterpret_cast<uint32_t *>(tile) + cc + (lane >> lg) * (stride >> 2);
    for (int y = lane >> lg; y < nrows; y += rstep, src += rstep * (W >> 2), dst += rstep * (stride >> 2)) *dst = __ldg(src);
  }
}

/* recompute output pixels [dx0,dx1] x [dy0,dy1] from the scratch and patch them into the frame: TX x TY taps in cv2's
 * order; surplus taps carry zero weights and may read scratch bytes outside the copied window (x + 0*b == x here).
 * CH: bytes per output pixel (3: `out` points at the channel's byte of pixel 0) */
template <int TX, int TY, int CH = 1>
__device__ __forceinline__ void tile_resolve(const uint8_t *tile, int stride, int wx0, int wy0, int dx0, int dx1, int dy0, int dy1, int dw,
                                             const TbxAreaPlan *__restrict__ plan, uint8_t *out, int lane) {
  const int ncol = dx1 - dx0 + 1;
  const int lg = ncol > 16 ? 5 : ncol > 8 ? 4 : ncol > 4 ? 3 : 2;
  const int c = lane & ((1 << lg) - 1), cpl = 1 << lg, rstep = 32 >> lg;
  for (int dxb = dx0; dxb <= dx1; dxb += cpl) {
    const int dx = dxb + c;
    const bool colok = dx <= dx1;
    const int dxc = colok ? dx : dx1;
    const uint8_t *col = tile + ((int)__ldg(&plan->xs0[dxc]) - wx0);
    float al[TX];
#pragma unroll
    for (int t = 0; t < TX; t++) al[t] = __ldg(&plan->xalpha[t][dxc]);
    for (int dy = dy0 + (lane >> lg); dy <= dy1; dy += rstep) {
      const uint8_t *row = col + ((int)__ldg(&plan->ys0[dy]) - wy0) * stride;
      float v = 0.0f;
#pragma unroll
      for (int k = 0; k < TY; k++) {
        float h = tbx_fmul(tbx_u8f(row[k * stride]), al[0]);
#pragma unroll
        for (int t = 1; t < TX; t++) h = tbx_fadd(h, tbx_fmul(tbx_u8f(row[k * stride + t]), al[t]));
        const float bh = tbx_fmul(__ldg(&plan->yalpha[k][dy]), h);
        v = k == 0 ? bh : tbx_fadd(v, bh);
      }
      const int iv = tbx_f2i_rn_small(v);
      if (colok) out[(dy * dw + dx) * CH] = (uint8_t)(iv < 0 ? 0 : iv > 255 ? 255 : iv);
    }
  }
}

/* dual mode: scratch <- max(scratch, scratch2) over the window, four pixels per operation */
__device__ __forceinline__ void tile_max(uint8_t *tile, const uint8_t *tile2, int stride, int wbytes, int nrows, int lane) {
  const int nwr = wbytes >> 2;
  const int lg = nwr > 16 ? 5 : nwr > 8 ? 4 : nwr > 4 ? 3 : 2;
  const int rstep = 32 >> lg;
  for (int cc = lane & ((1 << lg) - 1); cc < nwr; cc += 32)
    for (int y = lane >> lg; y < nrows; y += rstep) {
      uint32_t *p = reinterpret_cast<uint32_t *>(tile + y * stride) + cc;
      *p = __vmaxu4(*p, *(reinterpret_cast<const uint32_t *>(tile2 + y * stride) + cc));
    }
}

/* val: the byte painted (the entry's gray, or one component of its colour in RGB mode) */
__device__ __forceinline__ void paint_entry_coop(uint8_t *tile, int stride, int wx0, int wy0, int wx1, int wy1, const uint4 &q, uint32_t val, const uint32_t *R, int lane) {
  paint_tile(tile, stride, wx0, wy0, wx1, wy1, (int16_t)(q.x & 0xffffu), (int16_t)(q.x >> 16), (int16_t)(q.y & 0xffffu), (int16_t)(q.y >> 16),
             val, q.w, R, lane);
}

/* One tile row with more entries than the list holds: every tile of the row re-builds the primitives and paints
 * those that touch it, strictly in draw order (slow, but always correct).  CH = 3: once per channel, from the planar base
 * frames (channel c at bfr + c * W * H), into the interleaved frame.  DUAL_RGB: the dual RGB kernel's own copy -- ptxas
 * compiles a __noinline__ function once for all its callers, and that kernel has twice the registers of the others. */
template <int GAME, int TX, int TY, int CH = 1, bool DUAL_RGB = false>
__device__ __noinline__ void tile_row_rebuild(const uint32_t *R, const uint32_t *R2, const typename Traits<GAME>::Cfg &cfg, const typename Traits<GAME>::Table *tables,
                                              int base, int base2, const uint8_t *bfr, const uint8_t *bfr2, const TbxAreaPlan *__restrict__ plan, const TbxAreaPlan &cp,
                                              uint8_t *tile, uint8_t *tile2, int stride,
                                              int ty, int ths, int rA, int rB, int dyA, int dyB, uint8_t *out, int lane) {
  typedef Traits<GAME> T;
  constexpr int W = T::W, H = T::H;
  const int dw = cp.dw, dh = cp.dh;
  const int dy0 = ty << ths, dy1 = min(dy0 + (1 << ths) - 1, dh - 1);
  const int wy0 = cp.ys0[dy0], wy1 = min(H, (int)cp.ys0[dy1] + TY);
  for (int dxA = 0; dxA < dw; dxA += 16) {
    const int dxL = min(dxA + 15, dw - 1);
    const int wx0 = cp.xs0[dxA] & ~3, wx1 = min(W, ((int)cp.xs0[dxL] + TX + 3) & ~3);
#pragma unroll 1
    for (int ch = 0; ch < CH; ch++) {
    for (int st = 0; st < (R2 ? 2 : 1); st++) {
      const uint32_t *Rs = st ? R2 : R;
      const int bs = st ? base2 : base;
      uint8_t *ts = st ? tile2 : tile;
      tile_load<W>(ts, stride, (st ? bfr2 : bfr) + ch * (W * H), wx0, wy0, wx1, wy1, lane);
      __syncwarp();
      for (int g = 0; g < T::NG; g++) {
        int gb, ge, gmode;
        T::group(g, Rs, tables, bs, gb, ge, gmode);
          T::trim(g, Rs, cfg, bs, gb, ge);
        for (int s0 = gb; s0 < ge; s0 += 32) {
          const int s = s0 + lane;
          TbxPrim p = tbx_prim_none();
          if (s < ge) p = T::prim(Rs, cfg, tables, s, bs);
          uint4 e;
          uint32_t ext;
          bool hit = make_entry<W>(p, g, gmode, rA, rB, dyA, dyB, plan, e, ext);
          hit = hit && (int)(ext & 255u) <= dxL && (int)((ext >> 8) & 255u) >= dxA;
          unsigned m = __ballot_sync(0xffffffffu, hit);
          while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            uint4 q;
            q.x = __shfl_sync(0xffffffffu, e.x, l); q.y = __shfl_sync(0xffffffffu, e.y, l);
            q.z = __shfl_sync(0xffffffffu, e.z, l); q.w = __shfl_sync(0xffffffffu, e.w, l);
            const uint32_t val = CH == 1 ? q.z & 255u : (__shfl_sync(0xffffffffu, p.color, l) >> (8 * ch)) & 255u;
            paint_entry_coop(ts, stride, wx0, wy0, wx1, wy1, q, val, Rs, lane);
            __syncwarp();
          }
        }
      }
    }
    if (R2) { tile_max(tile, tile2, stride, wx1 - wx0, wy1 - wy0, lane); __syncwarp(); }
    tile_resolve<TX, TY, CH>(tile, stride, wx0, wy0, dxA, dxL, dy0, dy1, dw, plan, out + ch, lane);
    __syncwarp();
    }
  }
}

/* RGB (TBX_OBS_RGB_AREA): a.base[b] = planar base frame b (R, G, B planes of W x H), a.base_out[b] = its interleaved
 * down-sample, 3 bytes per output pixel; no HUD digit patches (they are gray) */
template <int GAME, int TX, int TY, bool DUAL, bool RGB = false>
__global__ void __launch_bounds__(TBX_TILE_THREADS, DUAL && RGB ? TBX_TILE_DUAL_RGB_MIN_CTAS : TBX_TILE_MIN_CTAS(TX, TY)) area_tile_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ typename Traits<GAME>::Cfg cfg_c,
                                                                         const __grid_constant__ TbxAreaPlan plan_c) {
  typedef Traits<GAME> T;
  constexpr int CH = RGB ? 3 : 1;
  constexpr int W = T::W, H = T::H, RW = T::RW;
  extern __shared__ uint4 smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>(smem_raw);
  uint32_t *recs = reinterpret_cast<uint32_t *>(smem);
  const typename T::Cfg &cfg = cfg_c;
  const typename T::Table *tables = (const typename T::Table *)a.tables;
  const TbxAreaPlan *__restrict__ plan = a.plan; /* per-lane indexed reads: global memory / L1 */
  const TbxAreaPlan &cp = plan_c;                /* warp-uniform reads: constant bank */
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarps = blockDim.x >> 5;
  constexpr bool dual = DUAL; /* observation = down-sample of max(frame of planes, frame of planes2): a.planes2 != NULL */
  uint32_t *recs2 = recs + RW * TBX_EPC;
  /* env-list mode (a.env_list != NULL: the envs the direct kernel of tbx_render_direct.cuh handed over): a small grid
   * walks the list chunk by chunk; otherwise CTA b renders envs 8b .. 8b+7 and the loop runs once */
  const int n_total = a.env_count ? *a.env_count : a.n;
  for (int chunk = blockIdx.x; chunk * TBX_EPC < n_total; chunk += gridDim.x) {
  const int e0 = chunk * TBX_EPC;
  const int ne = min(TBX_EPC, n_total - e0);
  if (chunk != (int)blockIdx.x) __syncthreads(); /* every warp is done with the previous chunk's records */
  for (int i = tid; i < RW * TBX_EPC; i += blockDim.x) {
    const int w = i / TBX_EPC, j = i - w * TBX_EPC;
    if (j < ne) {
      const int env = a.env_list ? a.env_list[e0 + j] : e0 + j;
      recs[j * RW + w] = a.planes[(size_t)w * a.n_pad + env];
      if (dual) recs2[j * RW + w] = a.planes2[(size_t)w * a.n_pad + env];
    }
  }
  __syncthreads(); /* the only CTA barrier per chunk: from here on every warp works alone */

  uint8_t *wmem = smem + a.smem_canvas + wid * a.warp_bytes;
  uint4 *list = reinterpret_cast<uint4 *>(wmem);
  uint32_t *exts = reinterpret_cast<uint32_t *>(wmem + TBX_TILE_LCAP * 16);
  uint32_t *tmask = exts + TBX_TILE_LCAP;
  uint32_t *cols = tmask + 8; /* RGB mode: each entry's colour (r | g << 8 | b << 16) */
  uint8_t *tile = reinterpret_cast<uint8_t *>(tmask + 8 + (RGB ? TBX_TILE_LCAP : 0));
  uint8_t *tile2 = tile + a.tile_bytes; /* dual mode: the second state's window */
  const int stride = a.tile_stride;
  constexpr int ths = TBX_TILE_HSHIFT;
  const int dw = cp.dw, dh = cp.dh, nty = (dh + (1 << ths) - 1) >> ths;
  const uint32_t lt_mask = (1u << lane) - 1u;

  for (int j = wid; j < ne; j += nwarps) {
    const uint32_t *R = recs + j * RW;
    const int base = T::base_id(R, cfg, tables);
    const uint8_t *bfr = base ? a.base[1] : a.base[0];
    const uint32_t *R2 = dual ? recs2 + j * RW : 0;
    const int base2 = dual ? T::base_id(R2, cfg, tables) : base;
    const uint8_t *bfr2 = base2 ? a.base[1] : a.base[0];
    const bool redo_all = base2 != base; /* the two frames differ everywhere the base frames do: recompute every tile */
    const int env = a.env_list ? a.env_list[e0 + j] : e0 + j;
    uint8_t *out = a.dst + (size_t)env * a.env_stride + (size_t)a.stack_slot * a.frame_bytes;
    { /* 1. the static part of the frame */
      const uint8_t *src = base ? a.base_out[1] : a.base_out[0];
      const int nb = dw * dh * CH;
      if ((a.frame_bytes & 15) == 0) {
        for (int i = lane; i < (nb >> 4); i += 32) reinterpret_cast<uint4 *>(out)[i] = __ldg(reinterpret_cast<const uint4 *>(src) + i);
      } else if ((a.frame_bytes & 3) == 0) {
        for (int i = lane; i < (nb >> 2); i += 32) reinterpret_cast<uint32_t *>(out)[i] = __ldg(reinterpret_cast<const uint32_t *>(src) + i);
      } else {
        for (int i = lane; i < nb; i += 32) out[i] = __ldg(src + i);
      }
    }
    __syncwarp(); /* orders the base copy before the patches other lanes write below */

    int nsw = 1;
    for (int sw = 0; sw < nsw; sw++) {
      /* this sweep: tile rows [tyA, tyB), output rows [dyA, dyB), source rows [rA, rB) */
      const int tyA = (sw * nty) / nsw, tyB = ((sw + 1) * nty) / nsw;
      if (tyA >= tyB) continue;
      const int dyA = tyA << ths, dyB = min(dh, tyB << ths);
      const int rA = cp.ys0[dyA], rB = min(H, (int)cp.ys0[dyB - 1] + TY);
      /* 2. build the sweep's list */
      __syncwarp();
      if (lane < 8) tmask[lane] = 0;
      __syncwarp();
      int n = 0;
      bool overflow = false;
      /* whole frame in one sweep: a digit's footprint is not clipped; dual mode: both frames on the same base frame */
      const bool use_patches = !RGB && a.patches[0] != 0 && nsw == 1 && (!dual || base == base2); /* the patches are gray */
      if constexpr (!dual) {
        for (int g = 0; g < T::NG && !overflow; g++) {
          int gb, ge, gmode;
          T::group(g, R, tables, base, gb, ge, gmode);
          T::trim(g, R, cfg, base, gb, ge);
          for (int s0 = gb; s0 < ge; s0 += 32) {
            const int s = s0 + lane;
            TbxPrim p = tbx_prim_none();
            if (s < ge) p = T::prim(R, cfg, tables, s, base);
            uint4 e;
            uint32_t ext;
            const bool ok = make_entry<W>(p, g, gmode, rA, rB, dyA, dyB, plan, e, ext);
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (m == 0) continue;
            if (n + __popc(m) > a.list_cap) { overflow = true; break; }
            if (ok) {
              const int slot = n + __popc(m & lt_mask);
              const int didx = T::digit_index(s);
              const bool cand = use_patches && didx >= 0 && p.bw == 3 && p.off < TBX_BANK_FONT + 50; /* a font sprite in a HUD digit slot */
              if (cand) e.z |= (TBX_ENTRY_DIGIT << 16) | ((uint32_t)didx << 24);
              list[slot] = e;
              exts[slot] = ext;
              if constexpr (RGB) cols[slot] = p.color;
              if (!cand) mark_tiles(tmask, ext, ths); /* candidates are marked below unless their patch can be used */
            }
            n += __popc(m);
          }
        }
      } else {
        /* Both states in one pass over the slots.  A slot whose primitive is the same in both states (HUD digits,
         * bricks, most sprites from one frame to the next) becomes ONE entry flagged 0x40 = "in both frames"; a run
         * hit by such entries only is rendered once.  Otherwise the slot emits its first-state entry, then its
         * second-state entry (flag 0x80): draw order is preserved within either state. */
        for (int g = 0; g < T::NG && !overflow; g++) {
          int gbA, geA, gmA, gbB, geB, gmB;
          T::group(g, R, tables, base, gbA, geA, gmA);
          T::trim(g, R, cfg, base, gbA, geA);
          T::group(g, R2, tables, base2, gbB, geB, gmB);
          T::trim(g, R2, cfg, base2, gbB, geB);
          const bool merge = base == base2 && gmA == gmB;
          const int lo = gbA >= geA ? gbB : gbB >= geB ? gbA : min(gbA, gbB), hi = max(geA, geB);
          for (int s0 = lo; s0 < hi; s0 += 32) {
            const int s = s0 + lane;
            TbxPrim pA = tbx_prim_none(), pB = tbx_prim_none();
            if (s >= gbA && s < geA) pA = T::prim(R, cfg, tables, s, base);
            if (s >= gbB && s < geB) pB = T::prim(R2, cfg, tables, s, base2);
            uint4 eA, eB;
            uint32_t xA, xB;
            const bool okA = make_entry<W>(pA, g, gmA, rA, rB, dyA, dyB, plan, eA, xA);
            const bool okB = make_entry<W>(pB, g | 0x80, gmB, rA, rB, dyA, dyB, plan, eB, xB);
            const bool both = merge && okA && okB && eA.x == eB.x && eA.y == eB.y && ((eA.z ^ eB.z) & 0xffu) == 0 && eA.w == eB.w &&
                              !(eA.w & TBX_PRIM_STATE) /* sprites stored in the record may differ bit by bit */
                              && (!RGB || pA.color == pB.color); /* RGB: two colours may share a gray */
            const unsigned m1 = __ballot_sync(0xffffffffu, okA), m2 = __ballot_sync(0xffffffffu, okB && !both);
            if ((m1 | m2) == 0) continue;
            if (n + __popc(m1) + __popc(m2) > a.list_cap) { overflow = true; break; }
            const int slot = n + __popc(m1 & lt_mask) + __popc(m2 & lt_mask);
            if (okA) {
              bool cand = false;
              if (both) {
                eA.z |= 0x40u << 8;
                const int didx = T::digit_index(s); /* the same HUD digit in both frames: a patch candidate (2b) */
                cand = use_patches && didx >= 0 && pA.bw == 3 && pA.off < TBX_BANK_FONT + 50;
                if (cand) eA.z |= (TBX_ENTRY_DIGIT << 16) | ((uint32_t)didx << 24);
              }
              list[slot] = eA;
              exts[slot] = xA;
              if constexpr (RGB) cols[slot] = pA.color;
              if (!cand) mark_tiles(tmask, xA, ths);
            }
            if (okB && !both) {
              list[slot + (okA ? 1 : 0)] = eB;
              exts[slot + (okA ? 1 : 0)] = xB;
              if constexpr (RGB) cols[slot + (okA ? 1 : 0)] = pB.color;
              mark_tiles(tmask, xB, ths);
            }
            n += __popc(m1) + __popc(m2);
          }
        }
      }
      if (overflow && nsw < nty) { /* halve the sweeps' height and start over (finished tiles are simply redone) */
        nsw = min(nty, nsw * 2);
        sw = -1;
        continue;
      }
      __syncwarp();

      if (overflow) {
        tile_row_rebuild<GAME, TX, TY, CH, DUAL && RGB>(R, R2, cfg, tables, base, base2, bfr, bfr2, plan, cp, tile, tile2, stride, tyA, ths, rA, rB, dyA, dyB, out, lane);
        continue;
      }
      /* 2b. HUD digits: a digit entry whose output rectangle meets no other entry's is the only thing that differs from
       * the base there, so its pre-resolved patch (host-built per slot and digit value, tbx_host.cpp) IS the result:
       * the entry leaves the list and the patch is copied after the tiles.  Others are marked like any entry. */
      uint32_t iso[TBX_TILE_LCAP / 32];
#pragma unroll
      for (int c = 0; c < TBX_TILE_LCAP / 32; c++) iso[c] = 0;
      if (use_patches) {
        const TbxDigitPatch *__restrict__ patches = base ? a.patches[1] : a.patches[0];
#pragma unroll
        for (int c = 0; c < TBX_TILE_LCAP / 32; c++) {
          if (c * 32 >= n) continue;
          const int i0 = c * 32 + lane;
          const bool cand = i0 < n && ((list[i0 < n ? i0 : 0].z >> 16) & TBX_ENTRY_DIGIT);
          unsigned candm = __ballot_sync(0xffffffffu, cand);
          if (n > 48) { /* a crowded frame (a wall full of holes): not worth the pairwise tests, mark the digits like any entry */
            if (cand) mark_tiles(tmask, exts[i0], ths);
            candm = 0;
          }
          while (candm) {
            const int l = __ffs(candm) - 1;
            candm &= candm - 1;
            const int i = c * 32 + l;
            const uint32_t xi = exts[i];
            const int xlo = xi & 255u, xhi = (xi >> 8) & 255u, ylo = (xi >> 16) & 255u, yhi = xi >> 24;
            bool ov = false;
            for (int j = lane; j < n; j += 32) {
              const uint32_t xj = exts[j];
              ov |= j != i && (int)(xj & 255u) <= xhi && (int)((xj >> 8) & 255u) >= xlo && (int)((xj >> 16) & 255u) <= yhi && (int)(xj >> 24) >= ylo;
            }
            const uint4 ei = list[i];
            const TbxDigitPatch *P = patches + ((ei.z >> 24) & 63u) * 10 + (ei.w & 0xffffu) / 5u;
            const bool usable = !__any_sync(0xffffffffu, ov) && __ldg(&P->w) != 0;
            if (usable) iso[c] |= 1u << l;
            else if (lane == 0) mark_tiles(tmask, xi, ths);
          }
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < TBX_TILE_LCAP / 32; c++)
          if ((iso[c] >> lane) & 1u) exts[c * 32 + lane] = 0x000000ffu; /* never hit: the tiles ignore it */
        __syncwarp();
      }
      if (redo_all) { /* every tile of the sweep, whether an entry touches it or not */
        __syncwarp();
        const uint32_t allcols = (1u << ((dw + 15) >> 4)) - 1u;
        if (lane < 8) {
          uint32_t mw = 0;
          for (int k = 0; k < 4; k++) { const int ty = lane * 4 + k; if (ty >= tyA && ty < tyB) mw |= allcols << (k * 8); }
          tmask[lane] = mw;
        }
        __syncwarp();
      } else if (n == 0) continue;

      /* 3. the marked tiles, one RUN of horizontally adjacent marked tiles of a tile row at a time.  Lanes hold the
       * extents of the entries (32 per chunk, one per lane), so "which entries feed this run, and which of its pixels" is one
       * compare per lane, a ballot and four warp reductions. */
      for (int ty = tyA; ty < tyB; ty++) {
        uint32_t rowbits = (tmask[ty >> 2] >> ((ty & 3) * 8)) & 0xffu;
        while (rowbits) {
          const int t0 = __ffs(rowbits) - 1;
          const int len = min(__ffs(~(rowbits >> t0)) - 1, TBX_TILE_MAX_RUN); /* consecutive marked tiles */
          rowbits &= ~(((1u << len) - 1u) << t0);
          const int rx0 = t0 * 16, rx1 = rx0 + len * 16 - 1, ry0 = ty << ths, ry1 = ry0 + (1 << ths) - 1;
          uint32_t hm[TBX_TILE_LCAP / 32];
          int bx0 = 255, bx1 = 0, by0 = 255, by1 = 0;
          bool two_frames = redo_all; /* dual mode: some hit entry belongs to one frame only (else both frames agree here) */
#pragma unroll
          for (int c = 0; c < TBX_TILE_LCAP / 32; c++) {
            hm[c] = 0;
            if (c * 32 >= n) continue;
            const uint32_t ext = c * 32 + lane < n ? exts[c * 32 + lane] : 0x000000ffu; /* 0xff: never hit */
            const int xlo = ext & 255u, xhi = (ext >> 8) & 255u, ylo = (ext >> 16) & 255u, yhi = ext >> 24;
            const bool hit = xlo <= rx1 && xhi >= rx0 && ylo <= ry1 && yhi >= ry0;
            hm[c] = __ballot_sync(0xffffffffu, hit);
            if (hit) { bx0 = min(bx0, xlo); bx1 = max(bx1, xhi); by0 = min(by0, ylo); by1 = max(by1, yhi); }
            if constexpr (dual) two_frames |= __ballot_sync(0xffffffffu, hit && !((list[c * 32 + lane].z >> 8) & 0x40u)) != 0;
          }
          int dx0 = max(rx0, __reduce_min_sync(0xffffffffu, bx0)), dx1 = min(rx1, __reduce_max_sync(0xffffffffu, bx1));
          int dy0 = max(ry0, __reduce_min_sync(0xffffffffu, by0)), dy1 = min(ry1, __reduce_max_sync(0xffffffffu, by1));
          if (redo_all) { dx0 = rx0; dx1 = min(rx1, dw - 1); dy0 = ry0; dy1 = min(ry1, dh - 1); }
          if (dx0 > dx1 || dy0 > dy1) continue;
          const int wx0 = cp.xs0[dx0] & ~3, wx1 = min(W, ((int)cp.xs0[dx1] + TX + 3) & ~3);
          const int wy0 = cp.ys0[dy0], wy1 = min(H, (int)cp.ys0[dy1] + TY);
          /* RGB mode: channel by channel through the same scratch window */
#pragma unroll 1
          for (int ch = 0; ch < CH; ch++) {
          tile_load<W>(tile, stride, bfr + ch * (W * H), wx0, wy0, wx1, wy1, lane);
          if (dual && two_frames) tile_load<W>(tile2, stride, bfr2 + ch * (W * H), wx0, wy0, wx1, wy1, lane);
          __syncwarp();
#pragma unroll
          for (int c = 0; c < TBX_TILE_LCAP / 32; c++) {
            uint32_t m = hm[c];
            if (m == 0) continue;
            uint4 e = make_uint4(0, 0, 0, 0);
            if ((m >> lane) & 1u) e = list[c * 32 + lane];
            while (m) {
              const int l = __ffs(m) - 1;
              const uint32_t zl = __shfl_sync(0xffffffffu, e.z, l);
              const bool st2 = (zl >> 15) & 1u; /* entry of the second state: its own scratch and record */
              const bool twice = dual && two_frames && ((zl >> 14) & 1u); /* in both frames: paint it into both windows */
              uint8_t *ts = st2 ? tile2 : tile;
              const uint32_t *Rs = st2 ? R2 : R;
              if (!((zl >> 16) & TBX_ENTRY_PAR)) { /* in-order group: one entry at a time */
                const uint4 q = list[c * 32 + l];
                const uint32_t qv = RGB ? (cols[c * 32 + l] >> (8 * ch)) & 255u : q.z & 255u;
                paint_entry_coop(ts, stride, wx0, wy0, wx1, wy1, q, qv, Rs, lane);
                if (twice) paint_entry_coop(tile2, stride, wx0, wy0, wx1, wy1, q, qv, R2, lane);
                __syncwarp();
                m &= m - 1;
                continue;
              }
              /* every hit entry of the same conflict-free group: the small solid ones lane-parallel, the rest one by one */
              const bool mine = ((m >> lane) & 1u) && ((e.z >> 8) & 255u) == ((zl >> 8) & 255u);
              const uint32_t same = __ballot_sync(0xffffffffu, mine);
              bool small = mine && ((e.z >> 16) & TBX_ENTRY_SMALL);
              uint32_t smalls = __ballot_sync(0xffffffffu, small);
              if (__popc(smalls) < 3) { smalls = 0; small = false; } /* too few to pay for one-lane loops: the warp paints each */
              uint32_t big = same & ~smalls;
              if (small) {
                const uint32_t ev = RGB ? (cols[c * 32 + lane] >> (8 * ch)) & 255u : e.z & 255u; /* the byte this lane's entry paints */
                paint_tile_lane(ts, stride, wx0, wy0, wx1, wy1, (int16_t)(e.x & 0xffffu), (int16_t)(e.x >> 16), (int16_t)(e.y & 0xffffu),
                                (int16_t)(e.y >> 16), ev);
                if (twice)
                  paint_tile_lane(tile2, stride, wx0, wy0, wx1, wy1, (int16_t)(e.x & 0xffffu), (int16_t)(e.x >> 16), (int16_t)(e.y & 0xffffu),
                                  (int16_t)(e.y >> 16), ev);
              }
              __syncwarp();
              while (big) {
                const int lb = __ffs(big) - 1;
                big &= big - 1;
                const uint4 q = list[c * 32 + lb];
                const uint32_t qv = RGB ? (cols[c * 32 + lb] >> (8 * ch)) & 255u : q.z & 255u;
                paint_entry_coop(ts, stride, wx0, wy0, wx1, wy1, q, qv, Rs, lane);
                if (twice) paint_entry_coop(tile2, stride, wx0, wy0, wx1, wy1, q, qv, R2, lane);
                __syncwarp();
              }
              m &= ~same;
            }
          }
          if (dual && two_frames) { tile_max(tile, tile2, stride, wx1 - wx0, wy1 - wy0, lane); __syncwarp(); }
          tile_resolve<TX, TY, CH>(tile, stride, wx0, wy0, dx0, dx1, dy0, dy1, dw, plan, out + ch, lane);
          __syncwarp(); /* the scratch canvas is overwritten by the next run or channel */
          }
        }
      }
      if (use_patches) { /* the isolated digits: their patches go in last (a run's bounding box may have swept over them) */
        const TbxDigitPatch *__restrict__ patches = base ? a.patches[1] : a.patches[0];
        __syncwarp();
#pragma unroll
        for (int c = 0; c < TBX_TILE_LCAP / 32; c++) {
          uint32_t m = iso[c];
          while (m) {
            const int i = c * 32 + __ffs(m) - 1;
            m &= m - 1;
            const uint4 ei = list[i];
            const TbxDigitPatch *P = patches + ((ei.z >> 24) & 63u) * 10 + (ei.w & 0xffffu) / 5u;
            const int px0 = __ldg(&P->x0), py0 = __ldg(&P->y0), pw = __ldg(&P->w), ph = __ldg(&P->h);
            const int cc = lane & 7;
            if (cc < pw)
              for (int r = lane >> 3; r < ph; r += 4) out[(py0 + r) * dw + px0 + cc] = __ldg(&P->px[r * pw + cc]);
          }
        }
      }
    }
    /* a reset observation and the rest of the env's ring: FrameStack.reset (atari_wrappers.py:262-266) fills every slot with
     * it; VecFrameStack (vec_env/vec_frame_stack.py:17-30) zeroes the stack and keeps the new frame only */
    if (a.reset_flags && a.stack_k > 1 && a.reset_flags[env]) {
      __syncwarp();
      uint8_t *ring = a.dst + (size_t)env * a.env_stride;
      const int nb = dw * dh * CH;
      const bool zero = a.stack_mode == 1;
      for (int k = 0; k < a.stack_k; k++) {
        if (k == a.stack_slot) continue;
        uint8_t *o2 = ring + (size_t)k * a.frame_bytes;
        if ((a.frame_bytes & 15) == 0) {
          for (int i = lane; i < (nb >> 4); i += 32) reinterpret_cast<uint4 *>(o2)[i] = zero ? make_uint4(0, 0, 0, 0) : __ldcg(reinterpret_cast<const uint4 *>(out) + i);
        } else {
          for (int i = lane; i < nb; i += 32) o2[i] = zero ? (uint8_t)0 : __ldcg(out + i);
        }
      }
    }
  }
  } /* chunk */
  /* env-list mode leaves the count as it is: the next render counts on the other one, and the direct kernel after it zeroes
   * this one (render_area) */
}

} /* namespace tbxk */
#endif
