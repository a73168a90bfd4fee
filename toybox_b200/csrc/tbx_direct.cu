/* tbx_direct.cu -- host side of the direct INTER_AREA kernels (tbx_render_direct.cuh): table upload and launcher.  A
 * translation unit of its own so that it compiles in parallel with, and rebuilds independently of, tbx_pool.cu. */
#include <mutex>
#include "tbx_render_direct.cuh"
#include <stdlib.h>
#include <vector>

using namespace tbxk;

static int align16(int v) { return (v + 15) & ~15; }

/* the tables a builder filled -> aux; nothing when the pair is outside its limits */
template <class D> static cudaError_t upload_direct(const std::vector<D> &A, Buf<uint8_t> &aux) {
  return A[0].ok ? aux.upload(reinterpret_cast<const uint8_t *>(A.data()), sizeof(D)) : cudaSuccess;
}

cudaError_t tbx_direct_build(const tbx::Config &c, const BrkTable *brk_default, const tbx::ResizeTab &rs, const TbxAreaPlan &plan, const uint8_t *base0_gray,
                             const uint8_t *base1_out, const TbxDigitPatch *patches1, Buf<uint8_t> &aux, Buf<uint8_t> &aux2) {
  if (c.game == TBX_BREAKOUT) {
    if (!brk_default) return cudaSuccess;
    std::vector<TbxBrkDirect> A(1);
    tbx::build_brk_direct(c, *brk_default, rs, plan, base0_gray, A[0]);
    if (!A[0].ok) return cudaSuccess;
    const Taps t = inst_taps(plan.tx, plan.ty); /* the kernel instantiation the image is laid out for */
    std::vector<uint8_t> img;
    tbx::build_brk_img(A[0], plan, t.x, t.y, base1_out, patches1, img);
    const cudaError_t e = upload_direct(A, aux);
    return e != cudaSuccess ? e : aux2.upload(img.data(), img.size());
  }
  if (c.game == TBX_AMIDAR) {
    std::vector<TbxAmiDirect> A(1);
    tbx::build_ami_direct(c, rs, plan, A[0]);
    return upload_direct(A, aux);
  }
  std::vector<TbxSiDirect> A(1);
  std::vector<TbxSpritePatch> patches;
  tbx::build_si_direct(c, rs, plan, base0_gray, A[0], patches);
  const cudaError_t e = upload_direct(A, aux);
  if (e != cudaSuccess || !aux || patches.empty()) return e;
  return aux2.upload(reinterpret_cast<const uint8_t *>(patches.data()), patches.size() * sizeof(TbxSpritePatch));
}

/* persistent grid: as many CTAs as the device keeps resident, each walks its share of the chunks.  The residency is cached per
 * (kernel, shared memory, device): the kernels share function-pointer types, so the cache is keyed by the pointer's value */
template <class K> static cudaError_t persistent_grid(K kernel, int smem, int n_chunks, int *grid_out) {
  struct Entry { const void *k; int smem, dev, resident; };
  static Entry cache[64];
  static int n_cache = 0;
  static std::mutex mu;
  int dev = 0;
  cudaGetDevice(&dev);
  int resident = 0;
  {
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < n_cache; i++)
      if (cache[i].k == (const void *)kernel && cache[i].smem == smem && cache[i].dev == dev) resident = cache[i].resident;
  }
  if (!resident) {
    int per_sm = 0, sms = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TBX_DIRECT_THREADS, smem);
    if (e != cudaSuccess) return e;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    resident = (per_sm > 0 ? per_sm : 1) * (sms > 0 ? sms : 148);
    std::lock_guard<std::mutex> lock(mu);
    if (n_cache < 64) cache[n_cache++] = Entry{(const void *)kernel, smem, dev, resident};
  }
  int grid = n_chunks < resident ? n_chunks : resident;
  if (const char *env = getenv("TBX_DIRECT_GRID")) if (atoi(env) > 0) grid = atoi(env) < n_chunks ? atoi(env) : n_chunks; /* tuning / tests */
  *grid_out = grid;
  return cudaSuccess;
}

/* the attribute is per device: set it on every launch (a cheap host-side call) rather than caching it per process */
template <class... P, class... A> static cudaError_t launch_persistent(void (*kernel)(P...), int smem, int n, cudaStream_t s, const A &...args) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  int grid = 1;
  e = persistent_grid(kernel, smem, (n + TBX_EPC - 1) / TBX_EPC, &grid);
  if (e != cudaSuccess) return e;
  kernel<<<grid, TBX_DIRECT_THREADS, smem, s>>>(args...);
  return cudaGetLastError();
}

cudaError_t tbx_launch_direct(const tbx::Config &c, const RenderArgs &a, const TbxAreaPlan &plan, DirectArgs d, size_t aux2_bytes, cudaStream_t s) {
  const int out_w = plan.dw, out_h = plan.dh;
  d.hstride = (out_w + 3) & ~3;
  d.smem_base = align16(out_w * out_h);
  return with_game(c.game, [&](auto g) {
    constexpr int G = decltype(g)::value, RW = Traits<G>::RW;
    if constexpr (G == TBX_BREAKOUT) {
      const int brk_rows = c.brk.n_rows < 1 || c.brk.n_rows > TBX_BRK_MAX_ROWS ? TBX_BRK_MAX_ROWS : c.brk.n_rows;
      /* the table image (tbx_direct.h) first; then two record stages per team; per warp the wall's H rows and the movers' records
       * (the env's record is read in place from its team's stage).  The image's size sets the residency, and with it the grid */
      if (aux2_bytes == 0 || aux2_bytes % 16 != 0 || aux2_bytes > 256 * 1024) return cudaErrorInvalidValue;
      d.smem_base = (int)aux2_bytes;
      d.warp_bytes = align16(brk_rows * d.hstride * (int)sizeof(float)) + 256;
      d.smem_total = d.smem_base + 2 * RW * TBX_EPC * 4 + (TBX_DIRECT_THREADS / 32) * d.warp_bytes;
      return with_taps<5>(plan.tx, plan.ty, [&](auto X, auto Y) {
        return launch_persistent(brk_direct_kernel<decltype(X)::value, decltype(Y)::value>, d.smem_total, a.n, s, a, c.brk, plan, d);
      });
    } else if constexpr (G == TBX_AMIDAR) {
      /* per warp: its env's record, the tile rows as looks, the movers' records; two record stages */
      d.warp_bytes = align16(RW * 4) + 256 + 448;
      d.smem_total = d.smem_base + 2 * RW * TBX_EPC * 4 + (TBX_DIRECT_THREADS / 32) * d.warp_bytes;
      return with_taps<4>(plan.tx, plan.ty, [&](auto X, auto Y) { /* three small per-pixel tables go behind the rest */
        return launch_persistent(ami_direct_kernel<decltype(X)::value, decltype(Y)::value>, d.smem_total + ami_tab_smem_bytes(out_h), a.n, s, a, plan, d);
      });
    } else {
      /* per warp: its env's record, the entries, two coverage bitmaps, the evaluated-entry list; one record stage */
      const int ow = (out_w + 31) / 32;
      d.warp_bytes = align16(RW * 4) + TBX_SD_MAX_ENTRIES * 32 + align16(2 * out_h * ow * 4) + TBX_SD_MAX_ENTRIES * 8;
      d.smem_total = d.smem_base + RW * TBX_EPC * 4 + (TBX_DIRECT_THREADS / 32) * d.warp_bytes;
      return with_taps<5>(plan.tx, plan.ty, [&](auto X, auto Y) { /* the plain-background map and the division table go behind the rest */
        return launch_persistent(si_direct_kernel<decltype(X)::value, decltype(Y)::value>, d.smem_total + si_tab_smem_bytes(out_w, out_h), a.n, s, a, plan, d);
      });
    }
  });
}

#ifdef TBX_SI_STATS
extern "C" int tbx_debug_si_stats(unsigned long long *out, int reset) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out, tbxk::d_si_stats, sizeof(unsigned long long) * 48) != cudaSuccess) return 1;
  if (reset) { unsigned long long z[48] = {0}; cudaMemcpyToSymbol(tbxk::d_si_stats, z, sizeof(z)); }
  return 0;
}
#endif
