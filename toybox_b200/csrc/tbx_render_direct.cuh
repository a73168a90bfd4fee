/* tbx_render_direct.cuh -- the DIRECT INTER_AREA kernels (84x84 gray WarpFrame observation): one warp per env, no
 * canvas, no draw list, no tiles.  See tbx_direct.h for the closed forms; this file is their warp-level schedule.
 *
 * Replaces get_state() + cv2.resize(INTER_AREA) (toybox/envs/atari/base.py:109, baselines/baselines/common/
 * atari_wrappers.py:243) for the envs the closed forms cover; the others are appended to a list that the general tile
 * kernel (tbx_render_area.cuh, env-list mode) renders right after.
 *
 * Breakout, per env (warp):
 *   1. frame <- pre-computed down-sample of base frame 1 (every brick alive), one bulk copy from shared memory;
 *   2. if a brick is dead: the wall's H rows (one look-up per brick row and output column) go to shared memory and the
 *      output words (4 pixels) x rows that a dead brick feeds are recomputed from them -- cost bounded by the wall's
 *      output area, whatever the number of holes;
 *   3. HUD digits: pre-resolved patches;
 *   4. paddle and balls: the output pixels their rectangles feed, their source windows built as packed bytes
 *      (base frame 0, brick grid, movers in draw order) and resolved in cv2's tap order.
 */
#ifndef TBX_RENDER_DIRECT_CUH
#define TBX_RENDER_DIRECT_CUH
#include "tbx_render_area.cuh"
#include "tbx_direct.h"
#include "tbx_direct_launch.h"

namespace tbxk {

#define TBX_DIRECT_THREADS 256
__host__ __device__ __forceinline__ int si_tab_smem_bytes(int dw, int dh) { return ((dh * ((dw + 31) >> 5) + 3) & ~3) * 4 + ((TBX_AREA_MAX_DST + 1 + 3) & ~3) * 4; }
__host__ __device__ __forceinline__ int ami_tab_smem_bytes(int dh) { return TBX_AMI_W + 256 + ((dh * 4 + 15) & ~15); }
__device__ __forceinline__ int brk_dig_cid(int slot) { return slot < 4 ? slot : slot >= TBX_MAX_DIGITS && slot < TBX_MAX_DIGITS + 2 ? slot - TBX_MAX_DIGITS + 4 : -1; }
#ifndef TBX_DIRECT_MIN_CTAS
#define TBX_DIRECT_MIN_CTAS 4
#endif

/* 16-byte asynchronous copies global -> shared (LDGSTS): the next chunk's records travel while this one is rendered */
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

/* PERSISTENT CTAs of two 4-warp TEAMS: a team renders chunks of 4 consecutive envs (one per warp), its first chunk fixed, the
 * next ones drawn from a device-wide counter.  Shared memory: the host-built IMAGE of every table the per-env code reads
 * (tbx_direct.h: the down-sample of base frame 1 -- every env's frame starts as ONE bulk shared -> global copy of it, cp.async.bulk,
 * no per-env load/store instructions --, the digit patches of the slots in use, base frame 0 by row classes, the plan's footprints,
 * weights and first-source indices, the brick grid, the wall's tables, a division table: L1 is too small next to this much shared
 * memory to keep sparse global tables), d.smem_base bytes loaded by one bulk copy per CTA; per team two stages of word-major
 * records (cp.async prefetch of the next chunk; a warp reads its env's record there, in place); per warp the wall's H rows and the
 * movers' records. */
template <int TX, int TY>
__global__ void __launch_bounds__(TBX_DIRECT_THREADS, TBX_DIRECT_MIN_CTAS) brk_direct_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ BrkCfg cfg_c,
                                                                            const __grid_constant__ TbxAreaPlan plan_c, const __grid_constant__ DirectArgs d) {
  constexpr int RW = TBX_WORDS(BrkRec);
  extern __shared__ uint4 smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>(smem_raw);
  const TbxBrkDirect *__restrict__ Ap = reinterpret_cast<const TbxBrkDirect *>(d.aux);
  const TbxBrkDirect &A = *Ap; /* warp-uniform scalars */
  const TbxAreaPlan &cp = plan_c;
  const int dw = cp.dw, dh = cp.dh, nrows = A.nrows;
  /* the image's regions (tbx_direct.h) */
  const TbxBrkImgLayout L = brk_img_layout(TX, TY, dw, dh, nrows, A.n_static, 0);
  const uint32_t *sdig = reinterpret_cast<const uint32_t *>(smem + TBX_BI_DIG);  /* [6 slots x 10 digits][13 words]: header + up to 48 pixels */
  const uint8_t *scls = smem + L.cls, *srowcls = smem + TBX_BI_ROWCLS;          /* base frame 0 by row classes */
  const uint32_t *sinv = reinterpret_cast<const uint32_t *>(smem + TBX_BI_INV);  /* inv32[] */
  const uint8_t *sxdlo = smem + TBX_BI_XDLO, *sxdhi = smem + TBX_BI_XDHI, *sydlo = smem + TBX_BI_YDLO, *sydhi = smem + TBX_BI_YDHI;
  const uint8_t *sxcol = smem + TBX_BI_XCOL, *syrow = smem + TBX_BI_YROW, *sbgray = smem + TBX_BI_BGRAY;
  const uint32_t *swordcols = reinterpret_cast<const uint32_t *>(smem + TBX_BI_WORDCOLS);
  const uint8_t *scol0 = smem + TBX_BI_COL0, *sdyrows = smem + TBX_BI_DYROWS, *shsel = smem + TBX_BI_HSEL; /* hsel: [dy][TY] */
  uint8_t *sbase = smem + TBX_BI_FIXED(TY);                                      /* base frame 1, down-sampled */
  const int ps = brk_plan_pitch(dw, dh);
  const float *sxa = reinterpret_cast<const float *>(smem + L.plan);             /* [TX][ps] */
  const float *sya = sxa + TX * ps;                                              /* [TY][ps] */
  const uint16_t *sxs = reinterpret_cast<const uint16_t *>(sya + TY * ps), *sys = sxs + ps; /* xs0, ys0 */
  const float *shlut = reinterpret_cast<const float *>(smem + L.hlut);           /* [brick row][2 alive bits][hstride]: the wall's H look-up */
  uint32_t *stage = reinterpret_cast<uint32_t *>(smem + d.smem_base);           /* [2 teams][2 stages][RW][4 envs] */
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uint8_t *wmem = smem + d.smem_base + 2 * RW * TBX_EPC * 4 + wid * d.warp_bytes;
  float *hw = reinterpret_cast<float *>(wmem);
  int4 *mrec = reinterpret_cast<int4 *>(wmem + d.warp_bytes - 256);             /* 3 x int4 per mover */
  /* two TEAMS of 4 warps per CTA, each with its own chunks of 4 envs (one 16-byte copy per state word), record stages and
   * barrier: a team waits for the slowest of 4 envs instead of 8 */
  constexpr int TEAM = 4, TEAM_THREADS = TEAM * 32;
  const int team = wid / TEAM, wt = wid % TEAM, ttid = tid % TEAM_THREADS;
  const int n_chunks = (a.n + TEAM - 1) / TEAM;
  const int nwords = dw >> 2, hs = d.hstride, nb = dw * dh;
  /* static rows of the wall's H sums, indexed by hsel's selector like the H rows: row sel - nrows of the image's hstatic */
  const float *shst = reinterpret_cast<const float *>(smem + L.hstatic) - nrows * hs;
  const bool bulk = (nb & 15) == 0 && (a.env_stride & 15) == 0 && (a.frame_bytes & 15) == 0;

  uint32_t *tstage = stage + team * 2 * RW * TEAM; /* [2][RW][4 envs] */
  auto prefetch = [&](int chunk, int st) {
    const uint32_t *src = a.planes + (size_t)chunk * TEAM;
    uint32_t *dst = tstage + st * RW * TEAM;
    for (int i = ttid; i < RW; i += TEAM_THREADS) cp_async16(dst + i * TEAM, src + (size_t)i * a.n_pad);
    cp_async_commit();
  };
  /* dynamic chunk scheduling: team (b, t) starts with chunk 2 b + t, further chunks come from a device-wide counter (the team's
   * first thread draws the id one iteration ahead; the barrier at the top of the loop publishes it), so the teams finish together
   * whatever their envs cost */
  __shared__ int s_next[2][2];
  __shared__ alignas(8) uint64_t s_img_bar; /* completes when the image has landed */
  const uint32_t img_bar = (uint32_t)__cvta_generic_to_shared(&s_img_bar);
  if (tid == 0) { /* the image: d.smem_base bytes at d.aux2, one bulk copy (well below the mbarrier's 2^20 - 1 transaction bytes) */
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(img_bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(img_bar), "r"(d.smem_base) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"((uint32_t)__cvta_generic_to_shared(smem)),
                 "l"(d.aux2), "r"(d.smem_base), "r"(img_bar) : "memory");
  }
  const int n_teams = (int)gridDim.x * (TBX_DIRECT_THREADS / TEAM_THREADS);
  if (ttid == 0) s_next[team][0] = n_teams + atomicAdd(d.sched, 1);
  if ((int)blockIdx.x * 2 + team < n_chunks) prefetch((int)blockIdx.x * 2 + team, 0);
  const int ok = A.ok, ncols = A.ncols, wdy0 = A.wdy0, wdy1 = A.wdy1, hud_dyhi = A.hud_dyhi, n_cls = A.n_cls;
  const int wy0 = A.wy0, wy1 = A.wy0 + nrows * A.bh;
  const uint32_t paddle_gray = A.paddle_gray, ball_gray = A.ball_gray;
  const TbxDigitPatch *__restrict__ patches = a.patches[1];
  __syncthreads(); /* the barrier is initialised */
  for (uint32_t img_in = 0; !img_in;)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }" : "=r"(img_in) : "r"(img_bar) : "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); /* the bulk copies below read sbase through the async proxy */
  const bool dig_smem = *reinterpret_cast<const int32_t *>(smem + TBX_BI_FLAGS) != 0;

  int st = 0, it = 0, nxt = 0;
  for (int chunk = (int)blockIdx.x * 2 + team; chunk < n_chunks; chunk = nxt, st ^= 1, it++) {
    cp_async_wait_all();
    asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(TEAM_THREADS) : "memory"); /* the team's barrier: this chunk's records have landed; its
                                                                                      * warps are done with the other stage; s_next[team][it & 1] is visible */
    nxt = s_next[team][it & 1];
    if (nxt < n_chunks) prefetch(nxt, st ^ 1);
    if (ttid == 0) s_next[team][(it + 1) & 1] = n_teams + atomicAdd(d.sched, 1);
    const int env = chunk * TEAM + wt;
    if (env >= a.n) continue;
    /* the env's record, read in place from the team's stage (word w at Rs[w * TEAM]): the stage is not written again before
     * the team's next barrier */
    const uint32_t *Rs = tstage + st * RW * TEAM + wt;
    const TbxAcc S{const_cast<uint32_t *>(Rs), TEAM};
    uint8_t *out = a.dst + (size_t)env * a.env_stride + (size_t)a.stack_slot * a.frame_bytes;
    /* movers: lane 0 the paddle, lanes 1..4 the balls; footprint = the output pixels the rectangle feeds */
    const TbxMover mine = brk_mover_rec(S, paddle_gray, ball_gray, lane < BRK_N_MOVERS ? lane : -1);
    const bool valid = mine.x0 < mine.x1;
    int fx0 = 0, fx1 = 0, fy0 = 0, fy1 = 0;
    if (valid) { fx0 = sxdlo[mine.x0]; fx1 = sxdhi[mine.x1 - 1]; fy0 = sydlo[mine.y0]; fy1 = sydhi[mine.y1 - 1]; }
    bool bad = valid && fy0 <= hud_dyhi;
    /* HUD digits: lanes 0..9 the score, 10..19 the lives */
    int dig = -1;
    const TbxDigitPatch *P = patches;
    if (lane < 2 * TBX_MAX_DIGITS && patches) {
      const int field = lane >= TBX_MAX_DIGITS;
      dig = tbx_digit_at(S.ldi(field ? TBX_HW(lives) : TBX_HW(score)), lane - field * TBX_MAX_DIGITS);
      if (dig >= 0) {
        const int cid = brk_dig_cid(lane);
        P = patches + lane * 10 + dig;
        bad |= (dig_smem && cid >= 0 ? (sdig[(cid * 10 + dig) * TBX_BRK_DIG_WORDS] >> 16) & 255u : (uint32_t)__ldg(&P->w)) == 0;
      }
    }
    const bool covered = ok && patches && S.ldi(TBX_HW(tbl)) == cfg_c.default_tbl;
    if (!covered || __any_sync(0xffffffffu, bad)) { /* the general kernel's */
      if (lane == 0) d.fb_list[atomicAdd(d.fb_count, 1)] = env;
      continue;
    }
    /* 1. every brick alive, nothing else: one bulk copy of the staged base frame, in flight while the warp prepares 2..4 */
    if (bulk) {
      if (lane == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out), "r"((uint32_t)__cvta_generic_to_shared(sbase)), "r"((uint32_t)nb) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    } else {
      for (int i = lane; i < (nb >> 2); i += 32) reinterpret_cast<uint32_t *>(out)[i] = reinterpret_cast<const uint32_t *>(sbase)[i];
    }
    /* 4a. paddle and balls, prepared while the base copy is in flight.  Lane m < 5 publishes its mover (rectangle, gray,
     * footprint) in the warp's shared memory; the footprints' output pixels form one list that the lanes share out 32 at
     * a time, whichever mover they belong to.  A pixel's TX x TY source window is built as packed bytes -- base frame 0
     * (two aligned word loads and a funnel shift per row), the brick grid where the window meets the wall, then every
     * mover's rectangle in draw order as a byte mask -- and resolved in cv2's tap order.  The first 32 pixels are computed
     * here and written in 4b, after the wall's and the HUD's. */
    const uint32_t vm = __ballot_sync(0xffffffffu, valid) & ((1u << BRK_N_MOVERS) - 1u);
    if (lane < BRK_N_MOVERS) {
      const int ncol = valid ? fx1 - fx0 + 1 : 0, nrow = valid ? fy1 - fy0 + 1 : 0;
      mrec[3 * lane + 0] = make_int4(mine.x0, mine.y0, mine.x1, mine.y1);
      mrec[3 * lane + 1] = make_int4((int)mine.gray * 0x01010101, fx0, fy0, ncol);
      mrec[3 * lane + 2] = make_int4(ncol * nrow, ncol > 1 ? (int)sinv[ncol] : 0, 0, 0);
    }
    __syncwarp();
    int total = 0;
#pragma unroll
    for (int m = 0; m < BRK_N_MOVERS; m++) total += mrec[3 * m + 2].x;
    const uint32_t *__restrict__ base0w = reinterpret_cast<const uint32_t *>(a.base[0]);
    const uint32_t *alive = Rs + BRK_W(alive) * TEAM; /* alive word k at alive[k * TEAM] */
    /* pixel p0 + lane of the movers' list: its offset in the frame (-1: past the end) and its value */
    auto mover_pixel = [&](int p0, int &o) -> uint32_t {
      const int l = p0 + lane;
      int mym = 0, myi = 0, off = 0;
#pragma unroll
      for (int m = 0; m < BRK_N_MOVERS; m++) {
        const int cnt = mrec[3 * m + 2].x;
        if (l >= off && l < off + cnt) { mym = m; myi = l - off; }
        off += cnt;
      }
      const bool act = l < total;
      const int4 f = mrec[3 * mym + 1];
      const int ncol = f.w, inv = mrec[3 * mym + 2].y;
      const int q = ncol > 1 ? (int)__umulhi((unsigned)myi, (unsigned)inv) : myi;
      const int dx = act ? f.y + myi - q * ncol : 0, dy = act ? f.z + q : 0;
      o = act ? dy * dw + dx : -1;
      const int xs = sxs[dx], ys = sys[dy];
      /* source rows as packed bytes: lo = taps 0..3, hi = tap 4 (TX == 5) */
      uint32_t lo[TY], hi[TY];
#pragma unroll
      for (int k = 0; k < TY; k++) {
        const int y = min(ys + k, TBX_BRK_H - 1); /* surplus taps carry zero weights: any in-frame pixel will do */
        /* the row of base frame 0: from its class in shared memory, or from the frame (both have 16 bytes of slack) */
        const uint32_t *rowp = n_cls ? reinterpret_cast<const uint32_t *>(scls + (int)srowcls[y] * TBX_BRK_W) : base0w + y * (TBX_BRK_W / 4);
        const uint32_t w0 = rowp[xs >> 2], w1 = rowp[(xs >> 2) + 1];
        lo[k] = __funnelshift_r(w0, w1, 8 * (xs & 3));
        hi[k] = 0;
        if (TX > 4) { const uint32_t w2 = rowp[(xs >> 2) + 2]; hi[k] = __funnelshift_r(w1, w2, 8 * (xs & 3)) & 255u; }
      }
      if (__any_sync(0xffffffffu, act && ys < wy1 && ys + TY > wy0)) { /* the brick grid */
        uint32_t cb[TX];
#pragma unroll
        for (int t = 0; t < TX; t++) cb[t] = sxcol[min(xs + t, TBX_BRK_W - 1)];
#pragma unroll
        for (int k = 0; k < TY; k++) {
          const uint32_t r = syrow[min(ys + k, TBX_BRK_H - 1)];
          if (r == 255u) continue;
#pragma unroll
          for (int t = 0; t < TX; t++) {
            if (cb[t] == 255u) continue;
            const uint32_t i = cb[t] * (uint32_t)nrows + r;
            if (!((alive[(i >> 5) * TEAM] >> (i & 31)) & 1u)) continue;
            const uint32_t g = sbgray[i];
            if (t < 4) lo[k] = (lo[k] & ~(255u << (8 * t))) | (g << (8 * t));
            else hi[k] = g;
          }
        }
      }
      uint32_t mleft = vm;
      while (mleft) { /* draw order: paddle, then the balls */
        const int m = __ffs(mleft) - 1;
        mleft &= mleft - 1;
        const int4 rc = mrec[3 * m];
        const uint32_t g4 = (uint32_t)mrec[3 * m + 1].x;
        const int ta = max(rc.x - xs, 0), tb = min(rc.z - xs, TX), ka = max(rc.y - ys, 0), kb = min(rc.w - ys, TY);
        if (ta >= tb || ka >= kb) continue;
        const uint32_t below_b = tb >= 4 ? 0xffffffffu : (1u << (8 * tb)) - 1u, below_a = ta >= 4 ? 0xffffffffu : (1u << (8 * ta)) - 1u;
        const uint32_t bm = below_b & ~below_a;
        const bool h5 = TX > 4 && ta <= 4 && tb > 4;
#pragma unroll
        for (int k = 0; k < TY; k++)
          if (k >= ka && k < kb) {
            lo[k] = (lo[k] & ~bm) | (g4 & bm);
            if (h5) hi[k] = g4 & 255u;
          }
      }
      float al[TX];
#pragma unroll
      for (int t = 0; t < TX; t++) al[t] = sxa[t * ps + dx];
      float acc = 0.0f;
#pragma unroll
      for (int k = 0; k < TY; k++) {
        float h = tbx_fmul(tbx_u8f(lo[k] & 255u), al[0]);
#pragma unroll
        for (int t = 1; t < TX; t++) h = tbx_fadd(h, tbx_fmul(tbx_u8f(t < 4 ? (lo[k] >> (8 * t)) & 255u : hi[k]), al[t]));
        const float bh = tbx_fmul(sya[k * ps + dy], h);
        acc = k == 0 ? bh : tbx_fadd(acc, bh);
      }
      const int iv = tbx_f2i_rn_small(acc);
      return (uint32_t)(iv > 255 ? 255 : iv); /* a sum of non-negative terms: never below zero */
    };
    int o_first = -1;
    uint32_t v_first = 0;
    if (total > 0) v_first = mover_pixel(0, o_first);
    /* 2. the wall */
    const uint32_t fullm = (1u << nrows) - 1u;
    const uint32_t colbits = lane < ncols ? brk_col_bits(S, BRK_W(alive), nrows, lane) : fullm;
    const uint32_t deadcols = __ballot_sync(0xffffffffu, colbits != fullm);
    bool landed = false; /* the base copy must have landed before the first patch is written over it */
#define TBX_DIRECT_LAND()                                                                       \
    if (!landed) {                                                                              \
      if (bulk && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");          \
      __syncwarp();                                                                             \
      landed = true;                                                                            \
    }
    if (deadcols) {
      const uint32_t deadrows = __reduce_or_sync(0xffffffffu, ~colbits & fullm);
      uint32_t rowmask[TBX_BRK_MAX_ROWS];
#pragma unroll
      for (int r = 0; r < TBX_BRK_MAX_ROWS; r++) rowmask[r] = __ballot_sync(0xffffffffu, (colbits >> r) & 1u);
      const uint32_t wmask = __ballot_sync(0xffffffffu, lane < nwords && (swordcols[lane] & deadcols));
      const uint32_t rmask = __ballot_sync(0xffffffffu, wdy0 + lane <= wdy1 && (sdyrows[wdy0 + lane] & deadrows));
      if (wmask && rmask) {
        const int wlo = __ffs(wmask) - 1, whi = 31 - __clz(wmask);
        __syncwarp(); /* the previous env's readers of the H rows are done */
        for (int dx = 4 * wlo + lane; dx < 4 * whi + 4; dx += 32) {
          const int c0 = scol0[dx];
#pragma unroll
          for (int r = 0; r < TBX_BRK_MAX_ROWS; r++)
            if (r < nrows) hw[r * hs + dx] = shlut[(r * 4 + ((rowmask[r] >> c0) & 3u)) * hs + dx];
        }
        __syncwarp();
        TBX_DIRECT_LAND();
        const int naw = __popc(wmask), rlo = wdy0 + __ffs(rmask) - 1, rhi = wdy0 + 31 - __clz(rmask);
        const int lg = naw > 16 ? 5 : naw > 8 ? 4 : naw > 4 ? 3 : naw > 2 ? 2 : naw > 1 ? 1 : 0;
        const int jw = lane & ((1 << lg) - 1), sub = lane >> lg, rpi = 32 >> lg;
        const int myword = jw < naw ? (int)__fns(wmask, 0, jw + 1) : -1;
        for (int dyb = rlo; dyb <= rhi; dyb += rpi) {
          const int dy = dyb + sub;
          if (myword < 0 || dy > rhi) continue;
          float acc[4];
#pragma unroll
          for (int k = 0; k < TY; k++) {
            const int sel = shsel[dy * TY + k];
            const float4 h = *reinterpret_cast<const float4 *>((sel < nrows ? hw : shst) + sel * hs + 4 * myword);
            const float b = sya[k * ps + dy];
            const float p0 = tbx_fmul(b, h.x), p1 = tbx_fmul(b, h.y), p2 = tbx_fmul(b, h.z), p3 = tbx_fmul(b, h.w);
            if (k == 0) { acc[0] = p0; acc[1] = p1; acc[2] = p2; acc[3] = p3; }
            else { acc[0] = tbx_fadd(acc[0], p0); acc[1] = tbx_fadd(acc[1], p1); acc[2] = tbx_fadd(acc[2], p2); acc[3] = tbx_fadd(acc[3], p3); }
          }
          uint32_t word = 0;
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const int iv = tbx_f2i_rn_small(acc[q]);
            word |= (uint32_t)(iv > 255 ? 255 : iv) << (8 * q); /* a sum of non-negative terms: never below zero */
          }
          *reinterpret_cast<uint32_t *>(out + dy * dw + 4 * myword) = word;
        }
      }
    }
    /* 3. HUD digits.  The slots cached in sdig (score digits 0..3, lives digits 0..1) in ONE pass over the concatenation of their
     * patches' pixels, lane l taking pixels l, l + 32, ...: the patches of two cached slots never share an output pixel at any
     * size this kernel accepts (tests/test_direct_digits_cpu.py), so their order does not matter.  The other shown digits come
     * after, one patch at a time from the table itself, in slot order: where one of them meets a cached slot it is the later
     * slot, as in the draw list. */
    TBX_DIRECT_LAND();
    {
      const int cid = brk_dig_cid(lane);
      const bool cached = dig >= 0 && dig_smem && cid >= 0;
      const uint32_t hdr = cached ? sdig[(cid * 10 + dig) * TBX_BRK_DIG_WORDS] : 0u; /* header word (x0, y0, w, h) */
      /* pixel offsets of the six slots in the concatenation (warp-uniform): slot c starts at off[c] */
      int off[TBX_BRK_DIG_SLOTS + 1];
      off[0] = 0;
#pragma unroll
      for (int c = 0; c < TBX_BRK_DIG_SLOTS; c++) {
        const uint32_t h = __shfl_sync(0xffffffffu, hdr, c < 4 ? c : TBX_MAX_DIGITS + c - 4);
        off[c + 1] = off[c] + (int)(((h >> 16) & 255u) * (h >> 24));
      }
      const int ntot = off[TBX_BRK_DIG_SLOTS];
      const uint8_t *sdigb = reinterpret_cast<const uint8_t *>(sdig);
      for (int i0 = 0; i0 < ntot; i0 += 32) {
        const int i = i0 + lane;
        int c = 0, o = 0;
#pragma unroll
        for (int k = 1; k < TBX_BRK_DIG_SLOTS; k++)
          if (i >= off[k]) { c = k; o = off[k]; } /* the last slot that starts at or before i: empty slots are skipped over */
        const int src = c < 4 ? c : TBX_MAX_DIGITS + c - 4;
        const uint32_t h = __shfl_sync(0xffffffffu, hdr, src);
        const int dg = __shfl_sync(0xffffffffu, dig, src);
        if (i < ntot) {
          const int q = i - o, pw = (h >> 16) & 255u;
          const int r = pw > 1 ? (int)__umulhi((unsigned)q, sinv[pw]) : q;
          out[(((h >> 8) & 255u) + r) * dw + (h & 255u) + q - r * pw] = sdigb[(c * 10 + dg) * TBX_BRK_DIG_WORDS * 4 + 4 + q];
        }
      }
      uint32_t dm = __ballot_sync(0xffffffffu, dig >= 0 && !cached);
      while (dm) {
        const int l = __ffs(dm) - 1;
        dm &= dm - 1;
        const int dgt = __shfl_sync(0xffffffffu, dig, l);
        const int cc = lane & 7;
        /* the patch: position, size, then w x h pixels */
        const TbxDigitPatch *Q = patches + l * 10 + dgt;
        const int px0 = __ldg(&Q->x0), py0 = __ldg(&Q->y0), pw = __ldg(&Q->w), ph = __ldg(&Q->h);
        if (cc < pw)
          for (int r = lane >> 3; r < ph; r += 4) out[(py0 + r) * dw + px0 + cc] = __ldg(&Q->px[r * pw + cc]);
      }
    }
    __syncwarp(); /* the movers' pixels go over the wall's */
    /* 4b. the movers' pixels */
    if (o_first >= 0) out[o_first] = (uint8_t)v_first;
    for (int p0 = 32; p0 < total; p0 += 32) {
      int o;
      const uint32_t v = mover_pixel(p0, o);
      if (o >= 0) out[o] = (uint8_t)v;
    }
  }
#undef TBX_DIRECT_LAND
  __syncthreads(); /* both teams have run dry */
  /* the last CTA to finish re-arms the chunk counter for the next launch, and zeroes the previous render's hand-over count (its
   * tile kernel ran before this launch): the next render appends to it */
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(d.sched + 1, 1) == (int)gridDim.x - 1) { d.sched[0] = 0; d.sched[1] = 0; *d.fb_other = 0; __threadfence(); }
  }
}

/* ------------------------------------------------------------------ Space Invaders: sparse sprites on a plain base
 * (tbx_direct.h).  Same persistent-CTA frame as the Breakout kernel: the base down-sample in shared memory, one bulk copy
 * of it per env, the records of a chunk staged word-major by cp.async (one stage: the next chunk is fetched as soon as
 * every warp has taken its record).  Per env (warp):
 *   1. the draw list's dynamic slots become ENTRIES in shared memory (clipped rectangle, gray, sprite reference, output
 *      footprint), three passes of 32 slots, in draw order;
 *   2. two bitmaps over the output pixels (covered once / covered twice) tell which entries share an output pixel with
 *      another one; an entry that does not, lies on plain background and has a pre-resolved patch (bank sprite in a usual
 *      colour, HUD digit) is a patch copy, one lane per entry;
 *   3. the other entries' footprints form a pixel list shared out 32 at a time; each pixel's TX x TY source window is built
 *      as packed bytes from base frame 0 and those entries in draw order (solid rectangles as byte masks, 16-bit sprites by
 *      shifting the row's bits under the window) and resolved in cv2's tap order. */
#define TBX_SI_DIRECT_MIN_CTAS 3
#define TBX_E_SPRITE_PATCH 1u
#define TBX_E_DIGIT_PATCH 2u
#define TBX_E_SCORE 4u /* a digit of the score: rendered with the others as one strip (TbxSiDirect.sc_px) */
#ifdef TBX_SI_STATS
__device__ unsigned long long d_si_stats[48];
#endif

template <int TX, int TY>
__global__ void __launch_bounds__(TBX_DIRECT_THREADS, TBX_SI_DIRECT_MIN_CTAS) si_direct_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ TbxAreaPlan plan_c,
                                                                                            const __grid_constant__ DirectArgs d) {
  constexpr int RW = TBX_WORDS(SiRec), W = TBX_SI_W, H = TBX_SI_H;
  constexpr int RECW_BYTES = (RW * 4 + 15) & ~15;
  extern __shared__ uint4 smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>(smem_raw);
  uint8_t *sbase = smem;
  uint32_t *stage = reinterpret_cast<uint32_t *>(smem + d.smem_base); /* [RW][8 envs] */
  const TbxSiDirect *__restrict__ Ap = reinterpret_cast<const TbxSiDirect *>(d.aux);
  const TbxSiDirect &A = *Ap;
  const TbxSpritePatch *__restrict__ spatch = reinterpret_cast<const TbxSpritePatch *>(d.aux2);
  const TbxDigitPatch *__restrict__ dpatch = a.patches[0];
  const TbxAreaPlan *__restrict__ plan = a.plan;
  const TbxAreaPlan &cp = plan_c;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int dw = cp.dw, dh = cp.dh, nb = dw * dh, ow = (dw + 31) >> 5; /* ow: bitmap words per output row */
  uint8_t *wmem = smem + d.smem_base + RW * TBX_EPC * 4 + wid * d.warp_bytes;
  uint32_t *recw = reinterpret_cast<uint32_t *>(wmem);
  int4 *ent = reinterpret_cast<int4 *>(wmem + RECW_BYTES);                       /* 2 x int4 per entry */
  uint32_t *occ1 = reinterpret_cast<uint32_t *>(ent + 2 * TBX_SD_MAX_ENTRIES);   /* [dh][ow]: covered by an entry */
  uint32_t *occ2 = occ1 + dh * ow;                                               /* covered by two or more */
  int *lst = reinterpret_cast<int *>(occ2 + dh * ow);                            /* evaluated entries: id, then pixel count */
  int *lcnt = lst + TBX_SD_MAX_ENTRIES;
  /* two small hot tables behind everything else (si_tab_smem_bytes: the launch adds them to d.smem_total) */
  uint32_t *splain = reinterpret_cast<uint32_t *>(smem + d.smem_total);          /* [dh][ow]: TbxSiDirect.plain */
  uint32_t *sinv = splain + ((dh * ow + 3) & ~3);                                /* inv32[] */
  const int n_chunks = (a.n + TBX_EPC - 1) / TBX_EPC;
  const bool bulk = (nb & 15) == 0 && (a.env_stride & 15) == 0 && (a.frame_bytes & 15) == 0;
  const int n_sets = A.n_sets, pxp = A.px_period, pyp = A.py_period;
  const uint32_t inv_px = A.inv_px, inv_py = A.inv_py;
  const int sc_ok = A.sc_ok, sc_gray = A.sc_gray, sc_dx0 = A.sc_dx0, sc_ncol = A.sc_ncol, sc_dy0 = A.sc_dy0, sc_nrow = A.sc_nrow;
  const uint32_t *__restrict__ base0w = reinterpret_cast<const uint32_t *>(a.base[0]);
  const uint32_t lt_mask = (1u << lane) - 1u;

  auto prefetch = [&](int chunk) {
    const uint32_t *src = a.planes + (size_t)chunk * TBX_EPC;
    for (int i = tid; i < RW * 2; i += TBX_DIRECT_THREADS) cp_async16(stage + i * 4, src + (size_t)(i >> 1) * a.n_pad + (i & 1) * 4);
    cp_async_commit();
  };
  __shared__ int s_next[2]; /* dynamic chunk scheduling, as in the Breakout kernel */
  if (tid == 0) s_next[0] = (int)gridDim.x + atomicAdd(d.sched, 1);
  if ((int)blockIdx.x < n_chunks) prefetch(blockIdx.x);
  for (int i = tid; i < ((nb + 15) >> 4); i += TBX_DIRECT_THREADS) reinterpret_cast<uint4 *>(sbase)[i] = __ldg(reinterpret_cast<const uint4 *>(a.base_out[0]) + i);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  for (int i = tid; i < dh * ow; i += TBX_DIRECT_THREADS) splain[i] = __ldg(&A.plain[i / ow][i % ow]);
  for (int i = tid; i <= TBX_AREA_MAX_DST; i += TBX_DIRECT_THREADS) sinv[i] = __ldg(&A.inv32[i]);
  const uint32_t *R = recw;

  int it = 0, nxt = 0;
  for (int chunk = blockIdx.x; chunk < n_chunks; chunk = nxt, it++) {
    cp_async_wait_all();
    __syncthreads(); /* the chunk's records have landed; every warp is done with its previous env; s_next[it & 1] is visible */
    nxt = s_next[it & 1];
    const int env = chunk * TBX_EPC + wid;
    if (env < a.n)
      for (int w = lane; w < RW; w += 32) recw[w] = stage[w * TBX_EPC + wid];
    __syncthreads(); /* the stage is free again */
    if (nxt < n_chunks) prefetch(nxt);
    if (tid == 0) s_next[(it + 1) & 1] = (int)gridDim.x + atomicAdd(d.sched, 1);
    if (env >= a.n) continue;
    uint8_t *out = a.dst + (size_t)env * a.env_stride + (size_t)a.stack_slot * a.frame_bytes;
    if (bulk) {
      if (lane == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out), "r"((uint32_t)__cvta_generic_to_shared(sbase)), "r"((uint32_t)nb) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    } else {
      for (int i = lane; i < (nb >> 2); i += 32) reinterpret_cast<uint32_t *>(out)[i] = reinterpret_cast<const uint32_t *>(sbase)[i];
    }
    /* 1. entries */
    for (int i = lane; i < 2 * dh * ow; i += 32) occ1[i] = 0;
    int n = 0, n_sc = 0, ufx0 = 255, ufx1 = -1, ufy0 = 255, ufy1 = -1; /* the score's digits as one strip: their count, their footprints' union */
    for (int s0 = SI_N_STATIC; s0 < SI_N_SLOTS; s0 += 32) {
      const int slot = s0 + lane;
      TbxPrim p = tbx_prim_none();
      if (slot < SI_N_SLOTS) p = si_prim(R, slot);
      const int x0 = max((int)p.x, 0), y0 = max((int)p.y, 0), x1 = min((int)p.x + (int)p.w, W), y1 = min((int)p.y + (int)p.h, H);
      const bool ok = p.h > 0 && x0 < x1 && y0 < y1;
      const unsigned m = __ballot_sync(0xffffffffu, ok);
      bool is_sc = false;
      int fx0 = 255, fx1 = -1, fy0 = 255, fy1 = -1;
      if (ok) {
        fx0 = __ldg(&plan->xdlo[x0]); fx1 = __ldg(&plan->xdhi[x1 - 1]); fy0 = __ldg(&plan->ydlo[y0]); fy1 = __ldg(&plan->ydhi[y1 - 1]);
        const uint32_t gray = tbx_luma(p.color);
        uint32_t kind = 0, ref = 0;
        const bool whole = p.x >= 0 && p.y >= 0 && (int)p.x + (int)p.w <= W && (int)p.y + (int)p.h <= H;
        if (sc_ok && whole && p.bw == 3 && slot < SI_SLOT_LIVES && p.off < TBX_BANK_FONT + 50 && (int)gray == sc_gray) { /* a digit of the score */
          kind = TBX_E_SCORE; is_sc = true;
        } else if (whole && p.bw == 3 && slot < SI_SLOT_SHIELDS && p.off < TBX_BANK_FONT + 50 && dpatch) { /* a HUD digit */
          ref = (uint32_t)(slot - SI_SLOT_SCORE) * 10u + p.off / 5u;
          if (__ldg(&dpatch[ref].w) != 0) kind = TBX_E_DIGIT_PATCH;
        } else if (whole && n_sets && p.bw == 16 && p.scale == 0x11 && !(p.off & TBX_PRIM_STATE) && p.off >= TBX_BANK_INVADER) { /* a bank sprite: is there a patch set for (sprite, gray)? */
          const int idx = p.off >= TBX_BANK_BOOM ? 8 + ((int)p.off - TBX_BANK_BOOM) / 10 : ((int)p.off - TBX_BANK_INVADER) / 10;
          const uint32_t cand = __ldg(reinterpret_cast<const uint32_t *>(A.set_lut[idx & 15]));
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const uint32_t s = (cand >> (8 * k)) & 255u;
            if (s != 255u && __ldg(&A.set_off[s]) == p.off && __ldg(&A.set_gray[s]) == gray && (int)__ldg(&A.set_h[s]) == (int)p.h) { kind = TBX_E_SPRITE_PATCH; ref = s; }
          }
        }
        const int e = n + __popc(m & lt_mask);
        ent[2 * e] = make_int4(x0 | (y0 << 16), x1 | (y1 << 16), (int)((uint16_t)p.x | ((uint32_t)(uint16_t)p.y << 16)), (int)(gray | (kind << 8) | (ref << 16)));
        ent[2 * e + 1] = make_int4((int)((uint32_t)p.off | ((uint32_t)p.bw << 16) | ((uint32_t)p.scale << 24)), fx0 | (fx1 << 8) | (fy0 << 16) | (fy1 << 24), 0, slot);
      }
      n += __popc(m);
      if (s0 == SI_N_STATIC && sc_ok) { /* the score's slots are among the first 32 */
        n_sc = __popc(__ballot_sync(0xffffffffu, is_sc));
        ufx0 = __reduce_min_sync(0xffffffffu, is_sc ? fx0 : 255); ufx1 = __reduce_max_sync(0xffffffffu, is_sc ? fx1 : -1);
        ufy0 = __reduce_min_sync(0xffffffffu, is_sc ? fy0 : 255); ufy1 = __reduce_max_sync(0xffffffffu, is_sc ? fy1 : -1);
      }
    }
    __syncwarp();
    /* 2. which entries share an output pixel with another one.  The score's digits count as ONE entry, the union of their footprints
     * (neighbouring digits always share a column: the strip table below knows every pair) */
    if (n_sc && lane <= ufy1 - ufy0) {
      const int r = ufy0 + lane;
      for (int w = ufx0 >> 5; w <= ufx1 >> 5; w++) {
        const uint32_t mask = (w == ufx0 >> 5 ? 0xffffffffu << (ufx0 & 31) : 0xffffffffu) & (w == ufx1 >> 5 ? 0xffffffffu >> (31 - (ufx1 & 31)) : 0xffffffffu);
        const uint32_t dup = atomicOr(&occ1[r * ow + w], mask) & mask;
        if (dup) atomicOr(&occ2[r * ow + w], dup);
      }
    }
    for (int e = lane; e < n; e += 32) {
      if ((((uint32_t)ent[2 * e].w >> 8) & 255u) == TBX_E_SCORE) continue;
      const uint32_t fp = (uint32_t)ent[2 * e + 1].y;
      const int fx0 = fp & 255u, fx1 = (fp >> 8) & 255u, fy0 = (fp >> 16) & 255u, fy1 = fp >> 24;
      for (int w = fx0 >> 5; w <= fx1 >> 5; w++) {
        const uint32_t mask = (w == fx0 >> 5 ? 0xffffffffu << (fx0 & 31) : 0xffffffffu) & (w == fx1 >> 5 ? 0xffffffffu >> (31 - (fx1 & 31)) : 0xffffffffu);
        for (int r = fy0; r <= fy1; r++) {
          const uint32_t dup = atomicOr(&occ1[r * ow + w], mask) & mask;
          if (dup) atomicOr(&occ2[r * ow + w], dup);
        }
      }
    }
    __syncwarp();
    bool sc_shared = false; /* something else touches the score's strip: its digits are then evaluated like any overlapping entries */
    if (n_sc) {
      bool hit = false;
      if (lane <= ufy1 - ufy0)
        for (int w = ufx0 >> 5; w <= ufx1 >> 5; w++) {
          const uint32_t mask = (w == ufx0 >> 5 ? 0xffffffffu << (ufx0 & 31) : 0xffffffffu) & (w == ufx1 >> 5 ? 0xffffffffu >> (31 - (ufx1 & 31)) : 0xffffffffu);
          hit |= (occ2[(ufy0 + lane) * ow + w] & mask) != 0;
        }
      sc_shared = __any_sync(0xffffffffu, hit);
    }
    int n_eval = 0, total = 0;
    bool any_shared = false;
    for (int e0 = 0; e0 < n; e0 += 32) {
      const int e = e0 + lane;
      bool patch = false, shared = false;
      int area = 0;
      if (e < n) {
        const uint32_t fp = (uint32_t)ent[2 * e + 1].y;
        const int fx0 = fp & 255u, fx1 = (fp >> 8) & 255u, fy0 = (fp >> 16) & 255u, fy1 = fp >> 24;
        area = (fx1 - fx0 + 1) * (fy1 - fy0 + 1);
        const uint32_t kind = ((uint32_t)ent[2 * e].w >> 8) & 255u;
        bool plain = true; /* sprite patches assume background around them; digit patches were resolved on the base itself */
        if (kind == TBX_E_SCORE) shared = sc_shared;
        else
        for (int w = fx0 >> 5; w <= fx1 >> 5 && !shared; w++) {
          const uint32_t mask = (w == fx0 >> 5 ? 0xffffffffu << (fx0 & 31) : 0xffffffffu) & (w == fx1 >> 5 ? 0xffffffffu >> (31 - (fx1 & 31)) : 0xffffffffu);
          for (int r = fy0; r <= fy1; r++) {
            if (occ2[r * ow + w] & mask) { shared = true; break; }
            if (kind == TBX_E_SPRITE_PATCH && (splain[r * ow + w] & mask) != mask) plain = false;
          }
        }
        patch = kind != 0 && !shared && plain;
        if (patch && kind != TBX_E_SCORE) ent[2 * e + 1].z = 1; /* rendered as a patch below (the score: as a strip) */
      }
      const unsigned em = __ballot_sync(0xffffffffu, e < n && !patch);
      if (e < n && !patch) { const int k = n_eval + __popc(em & lt_mask); lst[k] = e | (shared ? 0x10000 : 0); lcnt[k] = area; }
      n_eval += __popc(em);
      total += __reduce_add_sync(0xffffffffu, (e < n && !patch) ? area : 0);
      any_shared |= __any_sync(0xffffffffu, shared);
    }
#ifdef TBX_SI_STATS
    { /* tuning build: what the evaluated pixels are made of */
      if (lane == 0) { atomicAdd(&d_si_stats[0], 1ull); atomicAdd(&d_si_stats[1], (unsigned long long)n); atomicAdd(&d_si_stats[3], (unsigned long long)n_eval);
                       atomicAdd(&d_si_stats[4], (unsigned long long)total); atomicAdd(&d_si_stats[7], (unsigned long long)((total + 31) / 32)); }
      for (int k = lane; k < n_eval; k += 32) {
        const int id = lst[k] & 0xffff, conf = lst[k] >> 16, slot = ent[2 * id + 1].w;
        const int cls = slot < SI_SLOT_LIVES ? 0 : slot < SI_SLOT_SHIELDS ? 1 : slot < SI_SLOT_ENEMIES ? 2 : slot < SI_SLOT_SHIP ? 3 : slot == SI_SLOT_SHIP ? 4 : slot == SI_SLOT_UFO ? 5 : 6;
        atomicAdd(&d_si_stats[16 + cls], 1ull); atomicAdd(&d_si_stats[24 + cls], (unsigned long long)lcnt[k]);
        if (conf) { atomicAdd(&d_si_stats[5], 1ull); atomicAdd(&d_si_stats[6], (unsigned long long)lcnt[k]); atomicAdd(&d_si_stats[32 + cls], 1ull); }
      }
      for (int e = lane; e < n; e += 32) if (ent[2 * e + 1].z) atomicAdd(&d_si_stats[2], 1ull);
    }
#endif
    /* the base copy must have landed before anything is written over it */
    if (bulk && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncwarp();
    /* 2b. patches: one lane per entry */
    for (int e = lane; e < n; e += 32) {
      const int4 e1 = ent[2 * e + 1];
      if (!e1.z) continue;
      const int4 e0 = ent[2 * e];
      const uint32_t meta = (uint32_t)e0.w, kind = (meta >> 8) & 255u, ref = meta >> 16;
      const uint32_t fp = (uint32_t)e1.y;
      const int fx0 = fp & 255u, fy0 = (fp >> 16) & 255u;
      uint8_t *o = out + fy0 * dw + fx0;
      if (kind == TBX_E_SPRITE_PATCH) {
        const uint32_t ox = (uint32_t)(uint16_t)e0.z, oy = (uint32_t)e0.z >> 16; /* whole sprites: non-negative origin */
        const uint32_t xph = inv_px ? ox - __umulhi(ox, inv_px) * (uint32_t)pxp : 0u, yph = inv_py ? oy - __umulhi(oy, inv_py) * (uint32_t)pyp : 0u;
        const uint4 *P = reinterpret_cast<const uint4 *>(spatch + ((size_t)ref * pyp + yph) * pxp + xph);
        const uint4 q0 = __ldg(P), q1 = __ldg(P + 1);
        const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        const int pw = qw[0] & 255u, ph = (qw[0] >> 8) & 255u;
#pragma unroll
        for (int r = 0; r < TBX_SP_MAX_H; r++)
#pragma unroll
          for (int c = 0; c < TBX_SP_MAX_W; c++) {
            const int b = 2 + r * TBX_SP_MAX_W + c;
            if (r < ph && c < pw) o[r * dw + c] = (uint8_t)(qw[b >> 2] >> (8 * (b & 3)));
          }
      } else {
        const TbxDigitPatch *P = dpatch + ref;
        const int pw = __ldg(&P->w), ph = __ldg(&P->h);
        for (int r = 0; r < ph; r++)
          for (int c = 0; c < pw; c++) o[r * dw + c] = __ldg(&P->px[r * pw + c]);
      }
    }
    /* 2c. the score's strip: every pixel its digits feed, looked up by the digits of the (at most two) slots over its column */
    if (n_sc && !sc_shared) {
      const int ncu = ufx1 - ufx0 + 1, tot = ncu * (ufy1 - ufy0 + 1);
      const int32_t score = (int32_t)R[TBX_HW(score)];
      const uint32_t inv = ncu > 1 ? sinv[ncu] : 0u;
      for (int i = lane; i < tot; i += 32) {
        const int r = ncu > 1 ? (int)__umulhi((unsigned)i, inv) : i, c = i - r * ncu;
        const int dx = ufx0 + c, dy = ufy0 + r, tc = dx - sc_dx0, tr = dy - sc_dy0;
        if (tc < 0 || tc >= sc_ncol || tr < 0 || tr >= sc_nrow) continue;
        const int k0 = __ldg(&A.sc_slot[tc]);
        if (k0 == 255) continue;
        int da = tbx_digit_at(score, k0), db = k0 + 1 < TBX_MAX_DIGITS ? tbx_digit_at(score, k0 + 1) : -1;
        if (da < 0) da = 10;
        if (db < 0) db = 10;
        out[dy * dw + dx] = __ldg(&A.sc_px[tc][da][db][tr]);
      }
    }
    /* 3. the evaluated entries' pixels.  A pixel of an entry that shares no output pixel with another one sees that entry
     * only; pixels of entries that do are painted with every such entry, in draw order. */
    __syncwarp();
    for (int p0 = 0; p0 < total; p0 += 32) {
      const int l = p0 + lane;
      int myk = 0, myi = 0, off = 0;
      for (int k = 0; k < n_eval; k++) {
        const int cnt = lcnt[k];
        if (l >= off && l < off + cnt) { myk = k; myi = l - off; }
        off += cnt;
      }
      const bool act = l < total;
      const int mine = lst[myk];
      const bool conf = (mine >> 16) != 0;
      const uint32_t fp = (uint32_t)ent[2 * (mine & 0xffff) + 1].y;
      const int fx0 = fp & 255u, fx1 = (fp >> 8) & 255u, fy0 = (fp >> 16) & 255u;
      const int ncol = fx1 - fx0 + 1;
      const int q = ncol > 1 ? (int)__umulhi((unsigned)myi, sinv[ncol]) : myi;
      const int dx = act ? fx0 + myi - q * ncol : 0, dy = act ? fy0 + q : 0;
      const int xs = __ldg(&plan->xs0[dx]), ys = __ldg(&plan->ys0[dy]);
      uint32_t lo[TY], hi[TY];
#pragma unroll
      for (int k = 0; k < TY; k++) {
        const int y = min(ys + k, H - 1);
        const int ob = y * W + xs;
        const uint32_t w0 = __ldg(base0w + (ob >> 2)), w1 = __ldg(base0w + (ob >> 2) + 1);
        lo[k] = __funnelshift_r(w0, w1, 8 * (ob & 3));
        hi[k] = 0;
        if (TX > 4) { const uint32_t w2 = __ldg(base0w + (ob >> 2) + 2); hi[k] = __funnelshift_r(w1, w2, 8 * (ob & 3)) & 255u; }
      }
      /* paint entry `id` into this lane's window */
      auto paint = [&](int id) {
        const int4 e0 = ent[2 * id];
        const int x0 = e0.x & 0xffff, y0 = (uint32_t)e0.x >> 16, x1 = e0.y & 0xffff, y1 = (uint32_t)e0.y >> 16;
        const int ta = max(x0 - xs, 0), tb = min(x1 - xs, TX), ka = max(y0 - ys, 0), kb = min(y1 - ys, TY);
        if (ta >= tb || ka >= kb) return;
        const uint32_t spr = (uint32_t)ent[2 * id + 1].x;
        const uint32_t g = (uint32_t)e0.w & 255u, g4 = g * 0x01010101u;
        const int bw = (spr >> 16) & 255u;
        if (bw == 0) { /* a solid rectangle */
          const uint32_t below_b = tb >= 4 ? 0xffffffffu : (1u << (8 * tb)) - 1u, below_a = ta >= 4 ? 0xffffffffu : (1u << (8 * ta)) - 1u;
          const uint32_t bm = below_b & ~below_a;
          const bool h5 = TX > 4 && ta <= 4 && tb > 4;
#pragma unroll
          for (int k = 0; k < TY; k++)
            if (k >= ka && k < kb) { lo[k] = (lo[k] & ~bm) | (g4 & bm); if (h5) hi[k] = g; }
          return;
        }
        const int ox = (int16_t)(e0.z & 0xffff), oy = (int16_t)((uint32_t)e0.z >> 16);
        const uint32_t o = spr & 0xffffu;
        const bool in_state = (o & TBX_PRIM_STATE) != 0;
        const int ro = in_state ? (int)(o & 0x7fffu) : (int)o;
        const int sc = spr >> 24, sx = sc & 15, sy = sc >> 4;
        if (bw * sx <= 16) { /* at most 16 pixels per row (zoomed HUD digits included): shift the row's bits under the window */
          const int dd = xs - ox;
          const uint32_t iy = d_inv16[sy];
#pragma unroll
          for (int k = 0; k < TY; k++)
            if (k >= ka && k < kb) {
              const int py = ys + k - oy;
              const int ry = sy == 1 ? py : (int)(((uint32_t)py * iy) >> 16);
              const uint32_t bits = in_state ? R[ro + ry] : __ldg(&d_bank[ro + ry]);
              uint32_t row16; /* the row's pixels, left-aligned in 16 bits */
              if (sx == 1) row16 = bits << (16 - bw);
              else {
                row16 = 0;
                const uint32_t run = (1u << sx) - 1u;
                for (int j = 0; j < bw; j++)
                  if ((bits >> (bw - 1 - j)) & 1u) row16 |= run << (16 - (j + 1) * sx);
              }
              const uint32_t rev = __brev(row16 << 16); /* pixel q of the row at bit q */
              const uint32_t m5 = (dd >= 0 ? rev >> dd : rev << (-dd)) & 31u;
              const uint32_t bm = (((m5 & 15u) * 0x00204081u) & 0x01010101u) * 255u;
              lo[k] = (lo[k] & ~bm) | (g4 & bm);
              if (TX > 4 && (m5 & 16u)) hi[k] = g;
            }
          return;
        }
        /* wider zoomed sprites (none in the games' draw lists; interventions cannot create them either): tap by tap */
        const uint32_t ix = d_inv16[sx], iy = d_inv16[sy];
        for (int k = ka; k < kb; k++) {
          const int py = ys + k - oy;
          const int sy_i = sy == 1 ? py : (int)(((uint32_t)py * iy) >> 16);
          const uint32_t bits = in_state ? R[ro + sy_i] : __ldg(&d_bank[ro + sy_i]);
          uint32_t bm = 0;
          bool b5 = false;
          for (int t = ta; t < tb; t++) {
            const int px = xs + t - ox;
            const int sx_i = sx == 1 ? px : (int)(((uint32_t)px * ix) >> 16);
            if ((bits >> (bw - 1 - sx_i)) & 1u) { if (t < 4) bm |= 255u << (8 * t); else b5 = true; }
          }
#pragma unroll
          for (int kk = 0; kk < TY; kk++)
            if (kk == k) { lo[kk] = (lo[kk] & ~bm) | (g4 & bm); if (b5) hi[kk] = g; }
        }
      };
      if (act && !conf) paint(mine & 0xffff);
      if (any_shared && __any_sync(0xffffffffu, act && conf)) {
        for (int k2 = 0; k2 < n_eval; k2++) { /* draw order */
          const int id = lst[k2];
          if (!(id >> 16)) continue;
          if (act && conf) paint(id & 0xffff);
        }
      }
      float al[TX];
#pragma unroll
      for (int t = 0; t < TX; t++) al[t] = __ldg(&plan->xalpha[t][dx]);
      float acc = 0.0f;
#pragma unroll
      for (int k = 0; k < TY; k++) {
        float h = tbx_fmul(tbx_u8f(lo[k] & 255u), al[0]);
#pragma unroll
        for (int t = 1; t < TX; t++) h = tbx_fadd(h, tbx_fmul(tbx_u8f(t < 4 ? (lo[k] >> (8 * t)) & 255u : hi[k]), al[t]));
        const float bh = tbx_fmul(__ldg(&plan->yalpha[k][dy]), h);
        acc = k == 0 ? bh : tbx_fadd(acc, bh);
      }
      const int iv = tbx_f2i_rn_small(acc);
      if (act) out[dy * dw + dx] = (uint8_t)(iv > 255 ? 255 : iv);
    }
  }
  /* the last CTA to finish re-arms the chunk counter for the next launch */
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(d.sched + 1, 1) == (int)gridDim.x - 1) { d.sched[0] = 0; d.sched[1] = 0; __threadfence(); }
  }
}

/* ------------------------------------------------------------------ Amidar: the maze as a grid of looks (tbx_direct.h)
 * Same persistent frame as the Breakout kernel.  Per env (warp):
 *   1. frame <- down-sample of base frame 1 (the config board), one bulk copy;
 *   2. lane ty turns tile row ty into 2-bit looks (painted boxes fill their interior) and compares it with the board's: the
 *      output words x rows fed by a changed tile are recomputed -- horizontal sums by table look-up (two neighbouring looks and
 *      the output column), vertical taps over the tile rows; cost bounded by the maze's output area, however much is painted;
 *   3. HUD digits (score, lives, jumps): pre-resolved patches;
 *   4. enemies and player: the output pixels their 6 x 7 rectangles feed, source windows built from the tile looks. */
template <int TX, int TY>
__global__ void __launch_bounds__(TBX_DIRECT_THREADS, TBX_DIRECT_MIN_CTAS) ami_direct_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ TbxAreaPlan plan_c,
                                                                                          const __grid_constant__ DirectArgs d) {
  constexpr int RW = TBX_WORDS(AmiRec), W = TBX_AMI_W, H = TBX_AMI_H;
  constexpr int RECW_BYTES = (RW * 4 + 15) & ~15;
  extern __shared__ uint4 smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>(smem_raw);
  uint8_t *sbase = smem;
  uint32_t *stage = reinterpret_cast<uint32_t *>(smem + d.smem_base); /* [2][RW][8 envs] */
  const TbxAmiDirect *__restrict__ Ap = reinterpret_cast<const TbxAmiDirect *>(d.aux);
  const TbxAmiDirect &A = *Ap;
  const AmiTable *__restrict__ tables = reinterpret_cast<const AmiTable *>(a.tables);
  const TbxAreaPlan *__restrict__ plan = a.plan;
  const TbxAreaPlan &cp = plan_c;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uint8_t *wmem = smem + d.smem_base + 2 * RW * TBX_EPC * 4 + wid * d.warp_bytes;
  uint32_t *recw = reinterpret_cast<uint32_t *>(wmem);
  uint32_t *lk = reinterpret_cast<uint32_t *>(wmem + RECW_BYTES);             /* [31][2]: the tile rows as 2-bit looks */
  int4 *mrec = reinterpret_cast<int4 *>(wmem + RECW_BYTES + 256);             /* 3 x int4 per mover */
  /* three small per-pixel tables behind everything else (ami_tab_smem_bytes: the launch adds them to d.smem_total) */
  uint8_t *sxcol = smem + d.smem_total;                                       /* [W]: TbxAmiDirect.xcol */
  uint8_t *syrow = sxcol + TBX_AMI_W;                                         /* [H rounded up to 256]: yrow */
  uint32_t *sdyr = reinterpret_cast<uint32_t *>(syrow + 256);                 /* [dh]: dyrows */
  /* two teams of 4 warps per CTA, as in the Breakout kernel: own chunks of 4 envs, record stages and barrier */
  constexpr int TEAM = 4, TEAM_THREADS = TEAM * 32;
  const int team = wid / TEAM, wt = wid % TEAM, ttid = tid % TEAM_THREADS;
  const int n_chunks = (a.n + TEAM - 1) / TEAM;
  const int dw = cp.dw, dh = cp.dh, nwords = dw >> 2, nb = dw * dh;
  const bool bulk = (nb & 15) == 0 && (a.env_stride & 15) == 0 && (a.frame_bytes & 15) == 0;
  const int ok = A.ok, mdy0 = A.mdy0, mdy1 = A.mdy1, hud_dylo = A.hud_dylo;
  const uint32_t g0 = A.gray[0], player_gray = A.player_gray, enemy_gray = A.enemy_gray;
  const uint32_t glut = A.gray[0] | (A.gray[1] << 8) | (A.gray[2] << 16) | (A.gray[3] << 24); /* look -> gray, one byte each */
  const TbxDigitPatch *__restrict__ patches = a.patches[1];

  uint32_t *tstage = stage + team * 2 * RW * TEAM; /* [2][RW][4 envs] */
  auto prefetch = [&](int chunk, int st) {
    const uint32_t *src = a.planes + (size_t)chunk * TEAM;
    uint32_t *dst = tstage + st * RW * TEAM;
    for (int i = ttid; i < RW; i += TEAM_THREADS) cp_async16(dst + i * TEAM, src + (size_t)i * a.n_pad);
    cp_async_commit();
  };
  /* dynamic chunk scheduling per team (see the Breakout kernel) */
  __shared__ int s_next[2][2];
  const int n_teams = (int)gridDim.x * (TBX_DIRECT_THREADS / TEAM_THREADS);
  if (ttid == 0) s_next[team][0] = n_teams + atomicAdd(d.sched, 1);
  if ((int)blockIdx.x * 2 + team < n_chunks) prefetch((int)blockIdx.x * 2 + team, 0);
  for (int i = tid; i < ((nb + 15) >> 4); i += TBX_DIRECT_THREADS) reinterpret_cast<uint4 *>(sbase)[i] = __ldg(reinterpret_cast<const uint4 *>(a.base_out[1]) + i);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  for (int i = tid; i < W / 4; i += TBX_DIRECT_THREADS) reinterpret_cast<uint32_t *>(sxcol)[i] = __ldg(reinterpret_cast<const uint32_t *>(A.xcol) + i);
  for (int i = tid; i < 256 / 4; i += TBX_DIRECT_THREADS) reinterpret_cast<uint32_t *>(syrow)[i] = __ldg(reinterpret_cast<const uint32_t *>(A.yrow) + i);
  for (int i = tid; i < plan_c.dh; i += TBX_DIRECT_THREADS) sdyr[i] = __ldg(&A.dyrows[i]);
  const uint32_t *R = recw;
  __syncthreads(); /* the staged base frame and the tables are complete */

  int st = 0, it = 0, nxt = 0;
  for (int chunk = (int)blockIdx.x * 2 + team; chunk < n_chunks; chunk = nxt, st ^= 1, it++) {
    cp_async_wait_all();
    asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(TEAM_THREADS) : "memory"); /* the team's barrier */
    nxt = s_next[team][it & 1];
    if (nxt < n_chunks) prefetch(nxt, st ^ 1);
    if (ttid == 0) s_next[team][(it + 1) & 1] = n_teams + atomicAdd(d.sched, 1);
    const int env = chunk * TEAM + wt;
    if (env >= a.n) continue;
    {
      const uint32_t *src = tstage + st * RW * TEAM + wt;
      for (int w = lane; w < RW; w += 32) recw[w] = src[w * TEAM];
    }
    __syncwarp();
    uint8_t *out = a.dst + (size_t)env * a.env_stride + (size_t)a.stack_slot * a.frame_bytes;
    /* movers: lanes 0..7 the enemies, lane 8 the player (draw order) */
    TbxMover mine; mine.x0 = mine.y0 = mine.x1 = mine.y1 = 0; mine.gray = lane == TBX_AMI_MAX_ENEMIES ? player_gray : enemy_gray;
    if (lane < AMI_N_MOVERS) {
      const int m = lane == TBX_AMI_MAX_ENEMIES ? AMI_PLAYER : AMI_ENEMY(lane);
      const bool shown = lane == TBX_AMI_MAX_ENEMIES || (lane < (int32_t)R[AMI_W(n_enemies)] && !(int32_t)R[m + AMI_MW(caught)]);
      if (shown) {
        const int px = AMI_OFF_X + ami_floordiv((int32_t)R[m + AMI_MW(x)], 16) - 1, py = AMI_OFF_Y + ami_floordiv((int32_t)R[m + AMI_MW(y)], 16) - 1;
        const TbxPrim p = tbx_prim_rect(0, px, py, 6, 7); /* clamps far-away coordinates like the draw list does */
        if (p.h > 0) {
          mine.x0 = max((int)p.x, 0); mine.y0 = max((int)p.y, 0); mine.x1 = min((int)p.x + (int)p.w, W); mine.y1 = min((int)p.y + (int)p.h, H);
          if (mine.x0 >= mine.x1 || mine.y0 >= mine.y1) mine.x0 = mine.x1 = 0;
        }
      }
    }
    const bool valid = mine.x0 < mine.x1;
    int fx0 = 0, fx1 = 0, fy0 = 0, fy1 = 0;
    if (valid) { fx0 = __ldg(&plan->xdlo[mine.x0]); fx1 = __ldg(&plan->xdhi[mine.x1 - 1]); fy0 = __ldg(&plan->ydlo[mine.y0]); fy1 = __ldg(&plan->ydhi[mine.y1 - 1]); }
    bool bad = valid && fy1 >= hud_dylo;
    /* HUD digits: lanes 0..9 the score, 10..19 the lives, 20..29 the jumps */
    int dig = -1;
    const TbxDigitPatch *P = patches;
    if (lane < 3 * TBX_MAX_DIGITS && patches) {
      const int field = lane / TBX_MAX_DIGITS;
      const int32_t v = field == 0 ? (int32_t)R[TBX_HW(score)] : field == 1 ? (int32_t)R[TBX_HW(lives)] : (int32_t)R[AMI_W(jumps)];
      dig = tbx_digit_at(v, lane - field * TBX_MAX_DIGITS);
      if (dig >= 0) { P = patches + lane * 10 + dig; bad |= __ldg(&P->w) == 0; }
    }
    if (!ok || !patches || __any_sync(0xffffffffu, bad)) { /* the general kernel's */
      if (lane == 0) d.fb_list[atomicAdd(d.fb_count, 1)] = env;
      continue;
    }
    if (bulk) {
      if (lane == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out), "r"((uint32_t)__cvta_generic_to_shared(sbase)), "r"((uint32_t)nb) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    } else {
      for (int i = lane; i < (nb >> 2); i += 32) reinterpret_cast<uint32_t *>(out)[i] = reinterpret_cast<const uint32_t *>(sbase)[i];
    }
    /* 2. looks of tile row `lane`, and what differs from the config board */
    uint32_t l0 = 0, l1 = 0, d0 = 0, d1 = 0;
    if (lane < TBX_AMI_BH) {
      l0 = ami_looks_of_tags(R[AMI_W(tiles) + 2 * lane]);
      l1 = ami_looks_of_tags(R[AMI_W(tiles) + 2 * lane + 1]);
      uint32_t boxes = R[AMI_W(box_painted)];
      if (boxes) {
        const AmiTable &T = tables[(int32_t)R[TBX_HW(tbl)]];
        boxes &= __ldg(&T.all_boxes);
        while (boxes) { /* a painted box fills its interior, over whatever tiles lie there (draw order: boxes after tiles) */
          const int b = __ffs(boxes) - 1;
          boxes &= boxes - 1;
          const int tlx = __ldg(&T.tl_tx[b]), tly = __ldg(&T.tl_ty[b]), brx = __ldg(&T.br_tx[b]), bry = __ldg(&T.br_ty[b]);
          if (lane > tly && lane < bry && brx - tlx > 1) {
            const int ca = max(tlx + 1, 0), cb = min(brx - 1, TBX_AMI_BW - 1); /* tile columns ca..cb */
            if (ca <= cb) {
              const unsigned long long m64 = ((cb - ca + 1 >= 32 ? ~0ull : (1ull << (2 * (cb - ca + 1))) - 1ull)) << (2 * ca);
              l0 |= (uint32_t)m64; l1 |= (uint32_t)(m64 >> 32);
            }
          }
        }
      }
      d0 = l0 ^ __ldg(&A.base_looks[lane][0]);
      d1 = l1 ^ __ldg(&A.base_looks[lane][1]);
      d0 = (d0 | (d0 >> 1)) & 0x55555555u; d0 |= d0 << 1; /* both bits of a changed tile */
      d1 = (d1 | (d1 >> 1)) & 0x55555555u; d1 |= d1 << 1;
      lk[2 * lane] = l0; lk[2 * lane + 1] = l1;
    }
    const uint32_t rowsm = __ballot_sync(0xffffffffu, (d0 | d1) != 0);  /* tile rows with a changed tile */
    const uint32_t c0m = __reduce_or_sync(0xffffffffu, d0), c1m = __reduce_or_sync(0xffffffffu, d1); /* changed tile columns (look fields) */
    /* 4a. the movers, prepared while the base copy is in flight */
    const uint32_t vm = __ballot_sync(0xffffffffu, valid) & ((1u << AMI_N_MOVERS) - 1u);
    if (lane < AMI_N_MOVERS) {
      const int ncol = valid ? fx1 - fx0 + 1 : 0, nrow = valid ? fy1 - fy0 + 1 : 0;
      mrec[3 * lane + 0] = make_int4(mine.x0, mine.y0, mine.x1, mine.y1);
      mrec[3 * lane + 1] = make_int4((int)mine.gray * 0x01010101, fx0, fy0, ncol);
      mrec[3 * lane + 2] = make_int4(ncol * nrow, ncol > 1 ? (int)__ldg(&A.inv32[ncol]) : 0, 0, 0);
    }
    __syncwarp();
    /* which movers can reach the source windows of mover `lane`'s pixels (itself, and whoever walks next to it): a pixel paints those only */
    if (lane < AMI_N_MOVERS) {
      uint32_t near = 0;
      if (valid) {
        const int sx0 = __ldg(&plan->xs0[fx0]), sx1 = __ldg(&plan->xs0[fx1]) + TX, sy0 = __ldg(&plan->ys0[fy0]), sy1 = __ldg(&plan->ys0[fy1]) + TY;
#pragma unroll
        for (int m = 0; m < AMI_N_MOVERS; m++) {
          const int4 rc = mrec[3 * m];
          if (((vm >> m) & 1u) && rc.x < sx1 && rc.z > sx0 && rc.y < sy1 && rc.w > sy0) near |= 1u << m;
        }
      }
      mrec[3 * lane + 2].z = (int)near;
    }
    __syncwarp();
    int total = 0;
#pragma unroll
    for (int m = 0; m < AMI_N_MOVERS; m++) total += mrec[3 * m + 2].x;
    auto mover_pixel = [&](int p0, int &o) -> uint32_t {
      const int l = p0 + lane;
      int mym = 0, myi = 0, off = 0;
#pragma unroll
      for (int m = 0; m < AMI_N_MOVERS; m++) {
        const int cnt = mrec[3 * m + 2].x;
        if (l >= off && l < off + cnt) { mym = m; myi = l - off; }
        off += cnt;
      }
      const bool act = l < total;
      const int4 f = mrec[3 * mym + 1];
      const int ncol = f.w, inv = mrec[3 * mym + 2].y;
      const int q = ncol > 1 ? (int)__umulhi((unsigned)myi, (unsigned)inv) : myi;
      const int dx = act ? f.y + myi - q * ncol : 0, dy = act ? f.z + q : 0;
      o = act ? dy * dw + dx : -1;
      const int xs = __ldg(&plan->xs0[dx]), ys = __ldg(&plan->ys0[dy]);
      /* the source window from the tile looks: packed bytes, taps 0..3 of each row */
      uint32_t cb[TX], lo[TY];
#pragma unroll
      for (int t = 0; t < TX; t++) cb[t] = sxcol[min(xs + t, W - 1)];
#pragma unroll
      for (int k = 0; k < TY; k++) {
        const uint32_t r = syrow[min(ys + k, H - 1)];
        uint32_t row = g0 * 0x01010101u;
        if (r != 255u) {
          const uint32_t w0 = lk[2 * r], w1 = lk[2 * r + 1];
#pragma unroll
          for (int t = 0; t < TX; t++)
            if (cb[t] != 255u) {
              const uint32_t look = ((cb[t] < 16u ? w0 >> (2 * cb[t]) : w1 >> (2 * (cb[t] - 16u)))) & 3u;
              const uint32_t g = (glut >> (8 * look)) & 255u;
              row = (row & ~(255u << (8 * t))) | (g << (8 * t));
            }
        }
        lo[k] = row;
      }
      uint32_t mleft = (uint32_t)mrec[3 * mym + 2].z;
      while (mleft) { /* draw order: enemies, then the player */
        const int m = __ffs(mleft) - 1;
        mleft &= mleft - 1;
        const int4 rc = mrec[3 * m];
        const uint32_t g4 = (uint32_t)mrec[3 * m + 1].x;
        const int ta = max(rc.x - xs, 0), tb = min(rc.z - xs, TX), ka = max(rc.y - ys, 0), kb = min(rc.w - ys, TY);
        if (ta >= tb || ka >= kb) continue;
        const uint32_t below_b = tb >= 4 ? 0xffffffffu : (1u << (8 * tb)) - 1u, below_a = ta >= 4 ? 0xffffffffu : (1u << (8 * ta)) - 1u;
        const uint32_t bm = below_b & ~below_a;
#pragma unroll
        for (int k = 0; k < TY; k++)
          if (k >= ka && k < kb) lo[k] = (lo[k] & ~bm) | (g4 & bm);
      }
      float al[TX];
#pragma unroll
      for (int t = 0; t < TX; t++) al[t] = __ldg(&plan->xalpha[t][dx]);
      float acc = 0.0f;
#pragma unroll
      for (int k = 0; k < TY; k++) {
        float h = tbx_fmul(tbx_u8f(lo[k] & 255u), al[0]);
#pragma unroll
        for (int t = 1; t < TX; t++) h = tbx_fadd(h, tbx_fmul(tbx_u8f((lo[k] >> (8 * t)) & 255u), al[t]));
        const float bh = tbx_fmul(__ldg(&plan->yalpha[k][dy]), h);
        acc = k == 0 ? bh : tbx_fadd(acc, bh);
      }
      const int iv = tbx_f2i_rn_small(acc);
      return (uint32_t)(iv > 255 ? 255 : iv);
    };
    int o_first = -1;
    uint32_t v_first = 0;
    if (total > 0) v_first = mover_pixel(0, o_first);
    if (bulk && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncwarp(); /* the base copy has landed */
    /* 2b. the maze where it differs from the board */
    if (rowsm) {
      const uint32_t wmask = __ballot_sync(0xffffffffu, lane < nwords && ((__ldg(&A.wordcols[lane][0]) & c0m) | (__ldg(&A.wordcols[lane][1]) & c1m)) != 0);
      if (wmask) {
        const int naw = __popc(wmask);
        const int lg = naw > 16 ? 5 : naw > 8 ? 4 : naw > 4 ? 3 : naw > 2 ? 2 : naw > 1 ? 1 : 0;
        const int jw = lane & ((1 << lg) - 1), sub = lane >> lg, rpi = 32 >> lg;
        const int myword = jw < naw ? (int)__fns(wmask, 0, jw + 1) : -1;
        uint32_t c04 = 0;
        if (myword >= 0) c04 = __ldg(reinterpret_cast<const uint32_t *>(A.col0) + myword); /* col0 of the word's four columns */
        for (int dyb = mdy0; dyb <= mdy1; dyb += rpi) {
          const int dy = dyb + sub;
          const bool on = myword >= 0 && dy <= mdy1 && (sdyr[min(dy, dh - 1)] & rowsm) != 0;
          if (!on) continue;
          float acc[4];
#pragma unroll
          for (int k = 0; k < TY; k++) {
            const uint32_t r = __ldg(&A.ysel[dy][k]);
            const uint32_t w0 = r != 255u ? lk[2 * r] : 0u, w1 = r != 255u ? lk[2 * r + 1] : 0u;
            const float b = __ldg(&plan->yalpha[k][dy]);
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const uint32_t c0 = (c04 >> (8 * j)) & 255u;
              const uint32_t idx = (uint32_t)((((unsigned long long)w1 << 32) | w0) >> (2 * c0)) & 15u;
              const float p = tbx_fmul(b, __ldg(&A.hlut[idx][4 * myword + j]));
              acc[j] = k == 0 ? p : tbx_fadd(acc[j], p);
            }
          }
          uint32_t word = 0;
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const int iv = tbx_f2i_rn_small(acc[j]);
            word |= (uint32_t)(iv > 255 ? 255 : iv) << (8 * j);
          }
          *reinterpret_cast<uint32_t *>(out + dy * dw + 4 * myword) = word;
        }
      }
    }
    /* 3. HUD digits */
    {
      uint32_t dm = __ballot_sync(0xffffffffu, dig >= 0);
      while (dm) {
        const int l = __ffs(dm) - 1;
        dm &= dm - 1;
        const TbxDigitPatch *Q = reinterpret_cast<const TbxDigitPatch *>(__shfl_sync(0xffffffffu, (unsigned long long)P, l));
        const int px0 = __ldg(&Q->x0), py0 = __ldg(&Q->y0), pw = __ldg(&Q->w), ph = __ldg(&Q->h);
        const int cc = lane & 7;
        if (cc < pw)
          for (int r = lane >> 3; r < ph; r += 4) out[(py0 + r) * dw + px0 + cc] = __ldg(&Q->px[r * pw + cc]);
      }
    }
    __syncwarp(); /* the movers' pixels go over the maze's */
    /* 4b. the movers' pixels */
    if (o_first >= 0) out[o_first] = (uint8_t)v_first;
    for (int p0 = 32; p0 < total; p0 += 32) {
      int o;
      const uint32_t v = mover_pixel(p0, o);
      if (o >= 0) out[o] = (uint8_t)v;
    }
  }
  __syncthreads(); /* both teams have run dry */
  /* the last CTA to finish re-arms the chunk counter for the next launch, and zeroes the previous render's hand-over count (its
   * tile kernel ran before this launch): the next render appends to it */
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(d.sched + 1, 1) == (int)gridDim.x - 1) { d.sched[0] = 0; d.sched[1] = 0; *d.fb_other = 0; __threadfence(); }
  }
}

} /* namespace tbxk */
#endif
