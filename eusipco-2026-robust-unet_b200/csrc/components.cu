// Connected-component labelling, component statistics and small-region removal of water masks.
//
// rbu_label_components      labels int32 [B][H][W]: 0 background, components numbered 1..n in raster order of their first
//                           pixel (= scipy.ndimage.label with the 4- or 8-neighbour structure); counts int32 [B] = n.
// rbu_component_stats       per component: left, top, right, bottom, area, sum x, sum y (int64), from labels.
// rbu_remove_small_regions  water components below min_water become land, then land components of that result below
//                           min_land become water; uint8 0/1.
//
// Block-based union-find (Playne & Hawick 2018; Allegretti et al. 2019).  The root of a set is always its minimum
// per-image linear index y*W + x: a union links the larger root under the smaller one with atomicMin and retries from
// the value it displaced, so the final forest's roots do not depend on the order in which the atomics land.
//   local   one 32 x 32 CTA per tile: union-find in shared memory; parent[i] = the tile-local root (global index),
//           -1 for background; for the removal also area[local root] = the tile's pixel count of that root.
//   border  unions across the tile's top and left borders in global memory (8: also the diagonal pairs).  A border pixel
//           whose predecessor along the border is joined to the same neighbours inside both tiles skips its union.
//   flatten every pixel points at its root; the removal adds each tile-local root's area to the root (one atomic per
//           tile and component, never one per pixel); the labelling counts the roots per 64 row segments of 32 pixels.
//   scan    (labelling) one CTA per image: exclusive scan of the per-CTA root counts in raster order; counts_out.
//   rank    (labelling) each root gets its raster rank + 1, written into labels at the root's own position.
//   write   labels[i] = labels[root(i)];  removal: out = keep ? fg value : the other value.
// Per-image indices are int32 (H*W <= 2^30); every image offset is 64-bit.
#include <climits>

#include "components.cuh"

namespace {

constexpr int EW_THREADS = 256;                    // pixels per CTA of the write passes
constexpr int SCAN_THREADS = 1024;
constexpr int STATS_INIT_BLOCKS = 256;

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

bool dims_ok(int B, int H, int W) { return B >= 1 && B <= 65535 && H >= 1 && W >= 1 && H <= 32768 && W <= 32768; }

struct LabelLayout {                               // workspace of rbu_label_components (byte offsets)
  size_t parent, blk, total;
  int cx, nblk;                                    // segments per row, segment CTAs per image
};

LabelLayout label_layout(int B, int H, int W) {
  LabelLayout L;
  L.cx = rbu_cdiv(W, 32);
  L.nblk = rbu_cdiv((long)H * L.cx, SEGS);
  L.parent = 0;
  L.blk = align256((size_t)B * H * W * 4);
  L.total = align256(L.blk + (size_t)B * L.nblk * 4);
  return L;
}

struct RemoveLayout {                              // workspace of rbu_remove_small_regions
  size_t parent, area, total;
};

RemoveLayout remove_layout(int B, int H, int W) {
  RemoveLayout L;
  L.parent = 0;
  L.area = align256((size_t)B * H * W * 4);
  L.total = align256(L.area + (size_t)B * H * W * 4);
  return L;
}


// grid B: blk[b][*] becomes its exclusive scan; counts[b] = the total.
__global__ void __launch_bounds__(SCAN_THREADS)
cc_scan_kernel(int nblk, int* __restrict__ blk, int* __restrict__ counts) {
  __shared__ int wsum[32];
  int* v = blk + (long long)blockIdx.x * nblk;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int carry = 0;
  for (int base = 0; base < nblk; base += SCAN_THREADS) {
    const int i = base + threadIdx.x;
    const int x = i < nblk ? v[i] : 0;
    int incl = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    if (w == 0) {
      int s = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += n;
      }
      wsum[lane] = s;
    }
    __syncthreads();
    if (i < nblk) v[i] = carry + (w ? wsum[w - 1] : 0) + incl - x;
    carry += wsum[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) counts[blockIdx.x] = carry;
}

// labels[root] = 1 + the number of roots before it in raster order.
__global__ void __launch_bounds__(SEG_WARPS * 32)
cc_rank_kernel(int H, int W, int cx, const int* __restrict__ parent, const int* __restrict__ blk, int* __restrict__ labels) {
  __shared__ int segc[SEGS];
  const long long off = (long long)blockIdx.y * H * W;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned bal[SEGS_PER_WARP];
#pragma unroll
  for (int j = 0; j < SEGS_PER_WARP; ++j) {
    const int gi = seg_pixel(H, W, cx, j);
    bal[j] = __ballot_sync(0xffffffffu, gi >= 0 && parent[off + gi] == gi);
    if (lane == 0) segc[w * SEGS_PER_WARP + j] = __popc(bal[j]);
  }
  __syncthreads();
  if (w == 0) {                                      // exclusive scan of the 64 segment counts, two per lane
    const int a = segc[2 * lane], b = segc[2 * lane + 1];
    int incl = a + b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    segc[2 * lane] = incl - a - b;
    segc[2 * lane + 1] = incl - b;
  }
  __syncthreads();
  const int base = blk[(long long)blockIdx.y * gridDim.x + blockIdx.x];
  const unsigned lt = (1u << lane) - 1;
#pragma unroll
  for (int j = 0; j < SEGS_PER_WARP; ++j) {
    if (!((bal[j] >> lane) & 1)) continue;
    const int gi = seg_pixel(H, W, cx, j);
    labels[off + gi] = base + segc[w * SEGS_PER_WARP + j] + __popc(bal[j] & lt) + 1;
  }
}

// grid (ceil(H*W / 256), B): labels[i] = labels[root(i)] (0 for background); roots already hold their label.
__global__ void __launch_bounds__(EW_THREADS)
cc_label_write_kernel(int HW, const int* __restrict__ parent, int* __restrict__ labels) {
  const int i = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i >= HW) return;
  const long long off = (long long)blockIdx.y * HW;
  const int p = parent[off + i];
  if (p != i) labels[off + i] = p < 0 ? 0 : labels[off + p];
}

// grid (ceil(H*W / 256), B): out = fg_val where the pixel's component has at least min_area pixels, else 1 - fg_val.
__global__ void __launch_bounds__(EW_THREADS)
cc_keep_kernel(int HW, const int* __restrict__ parent, const int* __restrict__ area, int min_area, int fg_val,
               uint8_t* __restrict__ out) {
  const int i = blockIdx.x * EW_THREADS + threadIdx.x;
  if (i >= HW) return;
  const long long off = (long long)blockIdx.y * HW;
  const int p = parent[off + i];
  out[off + i] = (uint8_t)(p >= 0 && area[off + p] >= min_area ? fg_val : 1 - fg_val);
}

// ------------------------------------------------------------------------------------------------ statistics
// Rows [row_off[0], row_off[B]) of st = (left, top, right, bottom, area, sum x, sum y) = (max, max, -1, -1, 0, 0, 0).
__global__ void __launch_bounds__(256)
cc_stats_init_kernel(const long long* __restrict__ row_off, int B, long long* __restrict__ st) {
  const long long r1 = row_off[B];
  for (long long r = row_off[0] + (long long)blockIdx.x * 256 + threadIdx.x; r < r1; r += (long long)gridDim.x * 256) {
    long long* s = st + r * 7;
    s[0] = LLONG_MAX;
    s[1] = LLONG_MAX;
    s[2] = -1;
    s[3] = -1;
    s[4] = 0;
    s[5] = 0;
    s[6] = 0;
  }
}

// grid (ceil(W / 32), ceil(H / 32), B), block (32, 32): pixels of equal label that touch (8 neighbours) inside the tile
// form one group; the group's bounding box, area and coordinate sums go to row row_off[b] + label - 1 in one set of
// atomics.  Labels outside [1, row_off[b + 1] - row_off[b]] are ignored.
__global__ void __launch_bounds__(TILE * TILE)
cc_stats_kernel(const int* __restrict__ labels, int H, int W, const long long* __restrict__ row_off,
                long long* __restrict__ st) {
  __shared__ int key[TILE * TILE];
  __shared__ int lab[TILE * TILE];
  __shared__ int cnt[TILE * TILE], mnx[TILE * TILE], mxx[TILE * TILE], mny[TILE * TILE], mxy[TILE * TILE];
  __shared__ int sx[TILE * TILE], sy[TILE * TILE];
  const int lx = threadIdx.x, ly = threadIdx.y, li = ly * TILE + lx;
  const int x0 = blockIdx.x * TILE, y0 = blockIdx.y * TILE;
  const int x = x0 + lx, y = y0 + ly;
  const long long b = blockIdx.z;
  const long long first = row_off[b], rows = row_off[b + 1] - first;
  int k = 0;
  if (x < W && y < H) {
    k = labels[b * H * W + (long long)y * W + x];
    if (k < 1 || k > rows) k = 0;
  }
  key[li] = k;
  cnt[li] = 0;
  mnx[li] = INT_MAX;
  mxx[li] = -1;
  mny[li] = INT_MAX;
  mxy[li] = -1;
  sx[li] = 0;
  sy[li] = 0;
  const int r = tile_union_find(lab, key, lx, ly, 1);
  const unsigned grp = __match_any_sync(0xffffffffu, r);          // one warp = one tile row: y is uniform
  const int gmin = __reduce_min_sync(grp, lx), gmax = __reduce_max_sync(grp, lx);
  const int gsum = __reduce_add_sync(grp, lx), n = __popc(grp);
  if (r >= 0 && lx == __ffs(grp) - 1) {
    atomicAdd(&cnt[r], n);
    atomicMin(&mnx[r], gmin);
    atomicMax(&mxx[r], gmax);
    atomicMin(&mny[r], ly);
    atomicMax(&mxy[r], ly);
    atomicAdd(&sx[r], gsum);
    atomicAdd(&sy[r], n * ly);
  }
  __syncthreads();
  if (r != li) return;
  long long* s = st + (first + k - 1) * 7;
  const long long c = cnt[li];
  atomicMin(s + 0, (long long)(x0 + mnx[li]));
  atomicMin(s + 1, (long long)(y0 + mny[li]));
  atomicMax(s + 2, (long long)(x0 + mxx[li]));
  atomicMax(s + 3, (long long)(y0 + mxy[li]));
  atomicAdd(reinterpret_cast<unsigned long long*>(s + 4), (unsigned long long)c);
  atomicAdd(reinterpret_cast<unsigned long long*>(s + 5), (unsigned long long)(sx[li] + c * x0));
  atomicAdd(reinterpret_cast<unsigned long long*>(s + 6), (unsigned long long)(sy[li] + c * y0));
}


}  // namespace

extern "C" size_t rbu_label_workspace_bytes(int B, int H, int W) {
  if (!dims_ok(B, H, W)) return 0;
  return label_layout(B, H, W).total;
}

extern "C" int rbu_label_components(const void* mask, int kind, float threshold, int B, int H, int W, int connectivity,
                                    int32_t* labels_out, int32_t* counts_out, void* workspace, size_t workspace_bytes,
                                    void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(mask && labels_out && counts_out && workspace, "rbu_label_components: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_label_components: need 1 <= B <= 65535 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)",
                B, H, W);
  RBU_CHECK_ARG(kind == RBU_KIND_F32 || kind == RBU_KIND_U8, "rbu_label_components: kind must be RBU_KIND_F32 or RBU_KIND_U8");
  RBU_CHECK_ARG(connectivity == 4 || connectivity == 8, "rbu_label_components: connectivity must be 4 or 8 (got %d)",
                connectivity);
  RBU_CHECK_ARG(workspace_bytes >= rbu_label_workspace_bytes(B, H, W), "rbu_label_components: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "rbu_label_components: workspace must be 16-byte aligned");
  const LabelLayout L = label_layout(B, H, W);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* parent = reinterpret_cast<int*>(ws + L.parent);
  int* blk = reinterpret_cast<int*>(ws + L.blk);
  const int rc = union_find_passes<true, false>(mask, kind, threshold, 0, B, H, W, connectivity == 8, L.cx, L.nblk,
                                                parent, nullptr, blk, stream);
  if (rc != RBU_OK) return rc;
  cc_scan_kernel<<<B, SCAN_THREADS, 0, stream>>>(L.nblk, blk, counts_out);
  RBU_CHECK_LAUNCH();
  cc_rank_kernel<<<dim3(L.nblk, B), SEG_WARPS * 32, 0, stream>>>(H, W, L.cx, parent, blk, labels_out);
  RBU_CHECK_LAUNCH();
  cc_label_write_kernel<<<dim3(rbu_cdiv((long)H * W, EW_THREADS), B), EW_THREADS, 0, stream>>>(H * W, parent, labels_out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_component_stats(const int32_t* labels, int B, int H, int W, const int64_t* row_offsets,
                                   int64_t* stats_out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(labels && row_offsets && stats_out, "rbu_component_stats: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_component_stats: need 1 <= B <= 65535 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)",
                B, H, W);
  const long long* off = reinterpret_cast<const long long*>(row_offsets);
  long long* st = reinterpret_cast<long long*>(stats_out);
  cc_stats_init_kernel<<<STATS_INIT_BLOCKS, 256, 0, stream>>>(off, B, st);
  RBU_CHECK_LAUNCH();
  cc_stats_kernel<<<dim3(rbu_cdiv(W, TILE), rbu_cdiv(H, TILE), B), dim3(TILE, TILE), 0, stream>>>(labels, H, W, off, st);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" size_t rbu_remove_small_regions_workspace_bytes(int B, int H, int W) {
  if (!dims_ok(B, H, W)) return 0;
  return remove_layout(B, H, W).total;
}

extern "C" int rbu_remove_small_regions(const void* mask, int kind, float threshold, int B, int H, int W, int connectivity,
                                        int min_water, int min_land, uint8_t* out_u8, void* workspace,
                                        size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(mask && out_u8 && workspace, "rbu_remove_small_regions: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W),
                "rbu_remove_small_regions: need 1 <= B <= 65535 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)", B, H, W);
  RBU_CHECK_ARG(kind == RBU_KIND_F32 || kind == RBU_KIND_U8,
                "rbu_remove_small_regions: kind must be RBU_KIND_F32 or RBU_KIND_U8");
  RBU_CHECK_ARG(connectivity == 4 || connectivity == 8, "rbu_remove_small_regions: connectivity must be 4 or 8 (got %d)",
                connectivity);
  RBU_CHECK_ARG(min_water >= 0 && min_land >= 0, "rbu_remove_small_regions: min_water and min_land must be >= 0");
  RBU_CHECK_ARG(workspace_bytes >= rbu_remove_small_regions_workspace_bytes(B, H, W),
                "rbu_remove_small_regions: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "rbu_remove_small_regions: workspace must be 16-byte aligned");
  const RemoveLayout L = remove_layout(B, H, W);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* parent = reinterpret_cast<int*>(ws + L.parent);
  int* area = reinterpret_cast<int*>(ws + L.area);
  const int cx = rbu_cdiv(W, 32), nblk = rbu_cdiv((long)H * cx, SEGS), conn8 = connectivity == 8;
  const dim3 ew(rbu_cdiv((long)H * W, EW_THREADS), B);
  // step 1: water components below min_water become land (written to out_u8)
  int rc = union_find_passes<false, true>(mask, kind, threshold, 0, B, H, W, conn8, cx, nblk, parent, area, nullptr,
                                          stream);
  if (rc != RBU_OK) return rc;
  cc_keep_kernel<<<ew, EW_THREADS, 0, stream>>>(H * W, parent, area, min_water, 1, out_u8);
  RBU_CHECK_LAUNCH();
  // step 2: land components of that result below min_land become water
  rc = union_find_passes<false, true>(out_u8, RBU_KIND_U8, 0.f, 1, B, H, W, conn8, cx, nblk, parent, area, nullptr,
                                      stream);
  if (rc != RBU_OK) return rc;
  cc_keep_kernel<<<ew, EW_THREADS, 0, stream>>>(H * W, parent, area, min_land, 0, out_u8);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
