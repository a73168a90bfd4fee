/* tbx_direct_launch.h -- entry points of tbx_direct.cu (the direct INTER_AREA kernels, tbx_render_direct.cuh) for
 * tbx_pool.cu, and the host-side helpers both share.  Kept free of the kernel headers so that the two translation units
 * rebuild independently. */
#ifndef TBX_DIRECT_LAUNCH_H
#define TBX_DIRECT_LAUNCH_H
#include "tbx_render.cuh"
#include "tbx_host.h"
#include <type_traits>
#include <utility>

namespace tbxk {
struct DirectArgs {
  const void *aux;    /* the game's closed-form tables on the device (TbxBrkDirect, TbxSiDirect) */
  const void *aux2;   /* Space Invaders: the sprite patch tables (TbxSpritePatch[]) */
  int32_t *fb_list;   /* envs handed to the tile kernel */
  int *fb_count;
  int *sched;         /* [2]: next chunk id - grid size, finished CTAs (dynamic chunk scheduling of the persistent kernels) */
  int hstride;        /* floats per H row in shared memory */
  int warp_bytes;     /* shared memory per warp */
  int smem_base;      /* bytes of the staged base-frame down-sample at the start of shared memory */
  int smem_total;
};

/* An owning buffer of T elements in device memory (cudaMalloc) or pinned host memory (cudaMallocHost): move-only, freed
 * when it goes out of scope.  size() is the capacity in elements. */
template <class T, bool PINNED = false> class Buf {
  T *p_ = nullptr;
  size_t n_ = 0;

 public:
  Buf() = default;
  Buf(Buf &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
  Buf &operator=(Buf &&o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); return *this; }
  ~Buf() { reset(); }
  void reset() {
    if (p_) PINNED ? cudaFreeHost(p_) : cudaFree(p_);
    p_ = nullptr;
    n_ = 0;
  }
  T *get() const { return p_; }
  operator T *() const { return p_; }
  size_t size() const { return n_; }
  /* n elements, contents undefined; the buffer is empty when this fails */
  cudaError_t alloc(size_t n) {
    reset();
    void *q = nullptr;
    const cudaError_t e = PINNED ? cudaMallocHost(&q, n * sizeof(T)) : cudaMalloc(&q, n * sizeof(T));
    if (e == cudaSuccess) { p_ = (T *)q; n_ = n; }
    return e;
  }
  /* grow on demand: a new buffer of `cap` elements when this one holds fewer than `need` (contents are not kept) */
  cudaError_t grow(size_t need, size_t cap) { return need <= n_ ? cudaSuccess : alloc(cap); }
  cudaError_t grow(size_t need) { return grow(need, need); }
  /* n elements copied from the host */
  cudaError_t upload(const T *src, size_t n) {
    const cudaError_t e = alloc(n);
    return e != cudaSuccess ? e : cudaMemcpy(p_, src, n * sizeof(T), cudaMemcpyHostToDevice);
  }
};
template <class T> using PinnedBuf = Buf<T, true>;

template <int N> using Const = std::integral_constant<int, N>;

/* f(Const<GAME>()) for a pool's game id: the one place where a game id becomes a template argument */
template <class F> inline auto with_game(int game, F &&f) {
  if (game == TBX_BREAKOUT) return f(Const<TBX_BREAKOUT>());
  if (game == TBX_AMIDAR) return f(Const<TBX_AMIDAR>());
  return f(Const<TBX_SPACE_INVADERS>());
}

/* The tap counts (TX, TY) the INTER_AREA kernels are instantiated for: the smallest of 3/4/5 x 3/4 that covers a plan's
 * tx x ty taps, or 8 x 8 beyond 5 x 4 (the tile kernel only, single frames). */
struct Taps { int x, y; };
inline Taps inst_taps(int tx, int ty) {
  if (tx > 5 || ty > 4) return {8, 8};
  return {tx <= 3 ? 3 : tx <= 4 ? 4 : 5, ty <= 3 ? 3 : 4};
}
/* f(Const<TX>(), Const<TY>()) for inst_taps(tx, ty) with TX capped at MAX_TX: 8 x 8 is reached with MAX_TX = 8 only (the
 * direct kernels stop at 5 x 4, Amidar's at 4 x 4: its tables are built for tx <= 4) */
template <int MAX_TX, class F> inline auto with_taps(int tx, int ty, F &&f) {
  const Taps t = inst_taps(tx, ty);
  auto row = [&](auto X) { return t.y == 3 ? f(X, Const<3>()) : f(X, Const<4>()); };
  if constexpr (MAX_TX == 8) {
    if (t.x == 8) return f(Const<8>(), Const<8>());
  }
  if (t.x == 3) return row(Const<3>());
  if constexpr (MAX_TX == 4) {
    return row(Const<4>());
  } else {
    if (t.x == 4) return row(Const<4>());
    return row(Const<5>());
  }
}
}

/* closed-form tables of one (config, output size) pair on the device; aux stays empty when the pair is not covered */
cudaError_t tbx_direct_build(const tbx::Config &c, const BrkTable *brk_default, const tbx::ResizeTab &rs, const TbxAreaPlan &plan, const uint8_t *base0_gray,
                             tbxk::Buf<uint8_t> &aux, tbxk::Buf<uint8_t> &aux2);
/* the direct INTER_AREA kernel of the config's game for the plan's taps; d carries the tables and hand-over list, its
 * shared-memory layout is filled in here */
cudaError_t tbx_launch_direct(const tbx::Config &c, const tbxk::RenderArgs &a, const TbxAreaPlan &plan, tbxk::DirectArgs d, cudaStream_t s);
#endif
