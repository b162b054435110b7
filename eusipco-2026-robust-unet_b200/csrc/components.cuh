// Union-find passes shared by csrc/components.cu and csrc/contours.cu: the tile pass, the tile-border unions and
// the flatten pass of one foreground definition (see components.cu for the scheme).  A set's root is always its
// minimum per-image linear index y*W + x.
#pragma once

#include "rbu_common.cuh"

namespace {

constexpr int TILE = 32;                           // tile side of the local and border passes
constexpr int SEG_WARPS = 8;                       // warps per CTA of the segment passes
constexpr int SEGS_PER_WARP = 8;
constexpr int SEGS = SEG_WARPS * SEGS_PER_WARP;    // 32-pixel row segments per CTA: the unit of the raster-order scan

// Water: float32 p > threshold (strict), uint8 nonzero (the rules of rbu_coastline_stats' pred).
__device__ __forceinline__ bool is_water(const void* m, int kind, float thr, long long i) {
  if (kind == RBU_KIND_U8) return __ldg(static_cast<const uint8_t*>(m) + i) != 0;
  return __ldg(static_cast<const float*>(m) + i) > thr;
}

// Union-find on L (shared or global): roots satisfy L[r] == r; reads are volatile because other threads relink roots.
__device__ __forceinline__ int find_root(int* L, int x) {
  const volatile int* V = L;
  int p = V[x];
  while (p != x) {
    x = p;
    p = V[x];
  }
  return x;
}

__device__ __forceinline__ void unite(int* L, int a, int b) {
  bool done = false;
  do {
    a = find_root(L, a);
    b = find_root(L, b);
    if (a < b) {
      const int old = atomicMin(L + b, a);
      done = old == b;
      b = old;
    } else if (b < a) {
      const int old = atomicMin(L + a, b);
      done = old == a;
      a = old;
    } else {
      done = true;
    }
  } while (!done);
}

// The tile pass shared by the labelling, the removal and the statistics.  key[li] != 0 marks a foreground pixel; two
// neighbours join when their keys are equal.  Returns the tile-local root of the thread's pixel (-1 for background).
// A warp is a tile row: each run of equal keys starts out linked to its first pixel (a ballot), so only the rows
// need unions, and a pixel skips what the previous pixel of its run has joined (as the border pass does).
__device__ __forceinline__ int tile_union_find(int* lab, const int* key, int lx, int ly, int conn8) {
  const int li = ly * TILE + lx;
  __syncthreads();                                   // key[] is complete
  const int k = key[li];
  const bool left = k && lx > 0 && key[li - 1] == k;
  const unsigned starts = __ballot_sync(0xffffffffu, !left) & (0xffffffffu >> (TILE - 1 - lx));
  lab[li] = k ? ly * TILE + 31 - __clz(starts) : -1;
  __syncthreads();
  if (k && ly > 0) {
    const bool u = key[li - TILE] == k;
    if (!conn8) {
      if (u && !(left && key[li - TILE - 1] == k)) unite(lab, li, li - TILE);
    } else {
      if (!left) {                                   // else the previous pixel joined (ly - 1, lx - 2 .. lx)
        if (lx > 0 && key[li - TILE - 1] == k) unite(lab, li, li - TILE - 1);
        if (u) unite(lab, li, li - TILE);
      }
      if (lx < TILE - 1 && key[li - TILE + 1] == k && !u) unite(lab, li, li - TILE + 1);
    }
  }
  __syncthreads();
  return k ? find_root(lab, li) : -1;
}

// ------------------------------------------------------------------------------------------------ local pass
// grid (ceil(W / 32), ceil(H / 32), B), block (32, 32): foreground = water(mask) != invert.
template <bool AREA>
__global__ void __launch_bounds__(TILE * TILE)
cc_local_kernel(const void* __restrict__ mask, int kind, float thr, int invert, int H, int W, int conn8,
                int* __restrict__ parent, int* __restrict__ area) {
  __shared__ int key[TILE * TILE];
  __shared__ int lab[TILE * TILE];
  __shared__ int cnt[TILE * TILE];
  const int lx = threadIdx.x, ly = threadIdx.y, li = ly * TILE + lx;
  const int x0 = blockIdx.x * TILE, y0 = blockIdx.y * TILE;
  const int x = x0 + lx, y = y0 + ly;
  const bool in = x < W && y < H;
  const long long gi = (long long)blockIdx.z * H * W + (long long)y * W + x;
  key[li] = in && (is_water(mask, kind, thr, gi) != (invert != 0));
  if (AREA) cnt[li] = 0;
  const int r = tile_union_find(lab, key, lx, ly, conn8);
  if (AREA) {
    const unsigned grp = __match_any_sync(0xffffffffu, r);      // one warp = one tile row
    if (r >= 0 && lx == __ffs(grp) - 1) atomicAdd(&cnt[r], __popc(grp));
    __syncthreads();
  }
  if (!in) return;
  parent[gi] = r >= 0 ? (y0 + r / TILE) * W + x0 + r % TILE : -1;
  if (AREA) area[gi] = r == li ? cnt[li] : 0;
}

// ------------------------------------------------------------------------------------------------ border pass
// grid (ceil(W / 32), ceil(H / 32), B), 64 threads: threads 0-31 join the tile's top row to the row above, 32-63 its left
// column to the column on the left.  A pixel skips what its predecessor along the border has already joined: by
// induction every foreground border pixel ends up joined to all foreground pixels among its outside neighbours.
__global__ void __launch_bounds__(64)
cc_border_kernel(int H, int W, int conn8, int* __restrict__ parent) {
  int* P = parent + (long long)blockIdx.z * H * W;
  const int x0 = blockIdx.x * TILE, y0 = blockIdx.y * TILE;
  auto fg = [&](int i) { return P[i] >= 0; };
  if (threadIdx.x < 32) {
    const int t = threadIdx.x, x = x0 + t;
    if (y0 == 0 || x >= W) return;
    const int i = y0 * W + x;
    if (!fg(i)) return;
    const bool u = fg(i - W);
    if (!conn8) {
      if (u && !(t > 0 && fg(i - 1) && fg(i - W - 1))) unite(P, i, i - W);
      return;
    }
    const bool pred = t > 0 && fg(i - 1);            // (y0, x - 1) joined (y0 - 1, x - 2 .. x)
    if (!pred) {
      if (x > 0 && fg(i - W - 1)) unite(P, i, i - W - 1);
      if (u) unite(P, i, i - W);
    }
    if (x + 1 < W && fg(i - W + 1) && !(u && t < TILE - 1)) unite(P, i, i - W + 1);
  } else {
    const int t = threadIdx.x - 32, y = y0 + t;
    if (x0 == 0 || y >= H) return;
    const int i = y * W + x0;
    if (!fg(i)) return;
    const bool l = fg(i - 1);
    if (!conn8) {
      if (l && !(t > 0 && fg(i - W) && fg(i - W - 1))) unite(P, i, i - 1);
      return;
    }
    const bool pred = t > 0 && fg(i - W);            // (y - 1, x0) joined (y - 2 .. y, x0 - 1)
    if (!pred) {
      if (y > 0 && fg(i - W - 1)) unite(P, i, i - W - 1);
      if (l) unite(P, i, i - 1);
    }
    if (y + 1 < H && fg(i + W - 1) && !(l && t < TILE - 1)) unite(P, i, i + W - 1);
  }
}

// ------------------------------------------------------------------------------------------------ segment passes
// Segment s of an image covers row s / cx, columns 32 (s % cx) .. +31; CTA k of grid (nblk, B) covers segments
// [64k, 64k + 64), warp w the eight segments from 64k + 8w, one pixel per lane.
// The per-image index of this lane's pixel in the warp's j-th segment, -1 outside the image.
__device__ __forceinline__ int seg_pixel(int H, int W, int cx, int j) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long s = (long long)blockIdx.x * SEGS + w * SEGS_PER_WARP + j;
  if (s >= (long long)H * cx) return -1;
  const int y = (int)(s / cx), x = (int)(s % cx) * 32 + lane;
  return x < W ? y * W + x : -1;
}

// Flatten; COUNT: blk[b][k] = the roots in CTA k's segments; AREA: area[root] += area[local root].
template <bool COUNT, bool AREA>
__global__ void __launch_bounds__(SEG_WARPS * 32)
cc_flatten_kernel(int H, int W, int cx, int* __restrict__ parent, int* __restrict__ area, int* __restrict__ blk) {
  __shared__ int wsum[SEG_WARPS];
  const long long off = (long long)blockIdx.y * H * W;
  int* P = parent + off;
  int roots = 0;
  for (int j = 0; j < SEGS_PER_WARP; ++j) {
    const int gi = seg_pixel(H, W, cx, j);
    bool root = false;
    if (gi >= 0) {
      const int p = P[gi];
      if (p >= 0) {
        const int r = find_root(P, p);
        if (r != p) P[gi] = r;
        root = r == gi;
        if (AREA && r != gi) {
          const int a = area[off + gi];
          if (a) atomicAdd(area + off + r, a);
        }
      }
    }
    if (COUNT) roots += __popc(__ballot_sync(0xffffffffu, root));
  }
  if (COUNT) {
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = roots;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < SEG_WARPS; ++w) t += wsum[w];
      blk[(long long)blockIdx.y * gridDim.x + blockIdx.x] = t;
    }
  }
}

// local, border and flatten passes of one foreground definition (three launches).
template <bool COUNT, bool AREA>
int union_find_passes(const void* mask, int kind, float thr, int invert, int B, int H, int W, int conn8, int cx,
                      int nblk, int* parent, int* area, int* blk, cudaStream_t stream) {
  const dim3 tiles(rbu_cdiv(W, TILE), rbu_cdiv(H, TILE), B);
  cc_local_kernel<AREA><<<tiles, dim3(TILE, TILE), 0, stream>>>(mask, kind, thr, invert, H, W, conn8, parent, area);
  RBU_CHECK_LAUNCH();
  cc_border_kernel<<<tiles, 64, 0, stream>>>(H, W, conn8, parent);
  RBU_CHECK_LAUNCH();
  cc_flatten_kernel<COUNT, AREA><<<dim3(nblk, B), SEG_WARPS * 32, 0, stream>>>(H, W, cx, parent, area, blk);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

}  // namespace
