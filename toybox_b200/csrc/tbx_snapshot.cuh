/* tbx_snapshot.cuh -- the column copy behind device-resident state snapshots (tbx_state_save / tbx_state_load and
 * their wrapped-env forms).  A snapshot of k envs is uint32[rows][k], word-major like the pool's planes: column j is one
 * env's record, followed for a wrapped env by its 5 wrapper words.  One kernel serves every direction: entry j of a list
 * copies column src_idx[j] of the source to column dst_idx[j] of the destination, `rows` words.
 *
 * Mapping: lanes run over list entries, each thread copies a chunk of TBX_SNAP_ROWS rows (blockIdx.y picks the chunk), so
 * word r of 32 consecutive entries is one 128-byte line on the snapshot side, and on the plane side whenever the env ids
 * are ascending and contiguous (a full-pool save or load).  A thread issues all loads of its chunk before the stores.
 *
 * Every bound is checked before the memory it guards is touched: an entry whose source column, destination column or
 * (when tbl_lim >= 0) `tbl` word is out of range is skipped, and chunk 0 counts it once in *bad.  Destinations listed
 * more than once: `owner` (int32 per destination column, all -1 before snap_owner_kernel ran) holds the last valid entry
 * for each, and only that entry copies, so a destination receives one whole column, never a mix of two. */
#ifndef TBX_SNAPSHOT_CUH
#define TBX_SNAPSHOT_CUH
#include <cuda_runtime.h>
#include <stdint.h>

namespace tbxk {

#define TBX_SNAP_ROWS 16
#define TBX_SNAP_THREADS 256

/* one side of a copy: row r of column c is at (r < split ? base0 + r * stride : base1 + (r - split) * stride) + c.  Two
 * segments let the pool side of a wrapped env span its planes and its wrapper words; a snapshot is one segment
 * (base1 = base0 + split * stride). */
struct SnapSide {
  uint32_t *base0, *base1;
  size_t stride;
  int split;
  const int32_t *idx; /* column of entry j, NULL = j */
  int lim;            /* columns 0..lim-1 exist */
};

struct SnapArgs {
  SnapSide src, dst;
  int k, rows;
  int tbl_row;          /* row of hdr.tbl, or -1 (Space Invaders) */
  int tbl_lim;          /* >= 0: the source's tbl word must lie in 0..tbl_lim-1 (loads: the tables exported with it) */
  const int32_t *remap; /* may be NULL: tbl word -> remap[tbl] */
  int32_t *owner;       /* may be NULL: no destination can repeat */
  int *bad;
};

__device__ __forceinline__ uint32_t *snap_at(const SnapSide &s, int r, int c) {
  return (r < s.split ? s.base0 + (size_t)r * s.stride : s.base1 + (size_t)(r - s.split) * s.stride) + c;
}

/* the column pair of entry j, or false if any bound fails */
__device__ __forceinline__ bool snap_entry(const SnapArgs &a, int j, int &sc, int &dc) {
  sc = a.src.idx ? a.src.idx[j] : j;
  dc = a.dst.idx ? a.dst.idx[j] : j;
  if ((unsigned)sc >= (unsigned)a.src.lim || (unsigned)dc >= (unsigned)a.dst.lim) return false;
  if (a.tbl_row >= 0 && a.tbl_lim >= 0 && (unsigned)*snap_at(a.src, a.tbl_row, sc) >= (unsigned)a.tbl_lim) return false;
  return true;
}

/* pass 1 of a copy whose destinations may repeat: the last valid entry of each destination column wins */
__global__ void __launch_bounds__(TBX_SNAP_THREADS) snap_owner_kernel(SnapArgs a) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  int sc, dc;
  if (j < a.k && snap_entry(a, j, sc, dc)) atomicMax(a.owner + dc, j);
}

__global__ void __launch_bounds__(TBX_SNAP_THREADS) snap_copy_kernel(SnapArgs a) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.k) return;
  int sc, dc;
  if (!snap_entry(a, j, sc, dc)) {
    if (blockIdx.y == 0) atomicAdd(a.bad, 1);
    return;
  }
  if (a.owner && a.owner[dc] != j) return;
  const int r0 = blockIdx.y * TBX_SNAP_ROWS;
  uint32_t v[TBX_SNAP_ROWS];
#pragma unroll
  for (int i = 0; i < TBX_SNAP_ROWS; i++)
    if (r0 + i < a.rows) v[i] = *snap_at(a.src, r0 + i, sc);
#pragma unroll
  for (int i = 0; i < TBX_SNAP_ROWS; i++) {
    const int r = r0 + i;
    if (r >= a.rows) break;
    /* a remapped word was bounds-checked against tbl_lim in snap_entry (remap holds tbl_lim entries) */
    *snap_at(a.dst, r, dc) = (r == a.tbl_row && a.remap) ? (uint32_t)a.remap[v[i]] : v[i];
  }
}

} /* namespace tbxk */
#endif
