// Exact squared Euclidean distance transform (EDT) and coastline distance statistics.
//
// rbu_edt             D_F(y,x) = min over feature pixels (v,u) of (y-v)^2 + (x-u)^2, exact int32; -1 in an image with no
//                     feature pixel.  Equal to rint(scipy.ndimage.distance_transform_edt(F == 0) ** 2).
// rbu_coastline_stats the per-image, per-direction samples of the distances between the coastline of a predicted water
//                     mask and that of a target mask (DESIGN.md §8 item 8), reduced to exact integers and one float64 sum.
//
// The EDT is separable (Meijster et al. 2000) and takes a fixed number of passes whatever the distances:
//   1. mask   per (image, 64-row band, column): the band's feature rows as one 64-bit word (features read once).
//   2. carry  per (image, column): the last feature row above each band and the first one below it.
//   3. column per (image, band, column): g = the vertical distance to the nearest feature of the column (uint16, NONE if
//             the column has none), written TRANSPOSED, gT[image][x][y], through a shared-memory tile, so that
//   4. row    one thread per image row walks x with coalesced loads (adjacent threads = adjacent rows): the lower envelope
//             of the parabolas (x-u)^2 + g(u)^2 with Meijster's integer (int64) intersections, the stack in a workspace
//             laid out [x][y] so that adjacent threads touch adjacent words, and the output staged per 32 columns in
//             shared memory for coalesced int32 stores.
// The coastline statistics build both coastlines inline in pass 1 (no coastline image), run passes 2-4 on the 2B
// feature images, then reduce the samples: one pass for the counts, sums, maxima, tolerance counts and the top byte of a
// radix select, three more passes for the remaining bytes of the two order statistics of the 95th percentile, and one
// finalising block per (image, direction).  Every offset is 64-bit.
#include "rbu_common.cuh"

namespace {

constexpr int BAND = 64;                 // rows per band of the column pass (one 64-bit mask word)
constexpr uint16_t NONE = 0xffff;        // g of a column with no feature pixel (every real g is < 32768)
constexpr int COL_THREADS = 128;         // columns per block of the mask / column passes
constexpr int ST_THREADS = 256;          // columns per block of the statistics passes
constexpr int ST_BANDS = 8;              // bands per block of the statistics passes (the grid depends on H, W only)
constexpr int MAX_T = 8;

struct Layout {                          // EDT workspace of n images (byte offsets, 256-aligned)
  size_t mask, above, below, gT, stk, stt, total;
};

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

Layout edt_layout(long long n, int H, int W) {
  const long long nb = (H + BAND - 1) / BAND, Hp = nb * BAND;
  Layout L;
  L.mask = 0;
  L.above = align256(L.mask + (size_t)n * nb * W * 8);
  L.below = align256(L.above + (size_t)n * nb * W * 4);
  L.gT = align256(L.below + (size_t)n * nb * W * 4);
  L.stk = align256(L.gT + (size_t)n * W * Hp * 2);
  L.stt = align256(L.stk + (size_t)n * W * Hp * 4);
  L.total = align256(L.stt + (size_t)n * W * Hp * 2);
  return L;
}

// ------------------------------------------------------------------------------------------------ pass 1: band masks
// grid (ceil(W / 128), bands, images): bit r of mask[img][band][x] = features[img][band*64 + r][x] != 0
__global__ void __launch_bounds__(COL_THREADS)
edt_mask_kernel(const uint8_t* __restrict__ f, int H, int W, unsigned long long* __restrict__ mask) {
  const int x = blockIdx.x * COL_THREADS + threadIdx.x;
  if (x >= W) return;
  const long long img = blockIdx.z, nb = gridDim.y;
  const int y0 = blockIdx.y * BAND;
  const int rows = min(BAND, H - y0);
  const uint8_t* src = f + (img * H + y0) * (long long)W + x;
  unsigned long long m = 0;
  for (int r = 0; r < rows; ++r)
    if (__ldg(src + (long long)r * W)) m |= 1ull << r;
  mask[(img * nb + blockIdx.y) * W + x] = m;
}

// The water rules of rbu_coastline_stats: float32 pred p > threshold, float32 target t != 0, uint8 nonzero.
__device__ __forceinline__ bool water(const void* base, int kind, bool is_target, float thr, long long i) {
  if (kind == RBU_KIND_U8) return __ldg(static_cast<const uint8_t*>(base) + i) != 0;
  const float v = __ldg(static_cast<const float*>(base) + i);
  return is_target ? v != 0.f : v > thr;
}

// Coastline bit of (y, x): not water, and water among the four in-image neighbours.
__device__ __forceinline__ bool coast(const void* base, int kind, bool is_target, float thr, long long img_off, int H,
                                      int W, int y, int x) {
  const long long i = img_off + (long long)y * W + x;
  if (water(base, kind, is_target, thr, i)) return false;
  return (y > 0 && water(base, kind, is_target, thr, i - W)) || (y + 1 < H && water(base, kind, is_target, thr, i + W)) ||
         (x > 0 && water(base, kind, is_target, thr, i - 1)) || (x + 1 < W && water(base, kind, is_target, thr, i + 1));
}

// grid (ceil(W / 128), bands, B): band masks of P (image 2b, the coastline of pred) and G (image 2b + 1, of target).
__global__ void __launch_bounds__(COL_THREADS)
coast_mask_kernel(const void* __restrict__ pred, int pk, const void* __restrict__ target, int tk, float thr, int H, int W,
                  unsigned long long* __restrict__ mask) {
  const int x = blockIdx.x * COL_THREADS + threadIdx.x;
  if (x >= W) return;
  const long long b = blockIdx.z, nb = gridDim.y;
  const long long off = b * H * (long long)W;
  const int y0 = blockIdx.y * BAND;
  const int rows = min(BAND, H - y0);
  unsigned long long mp = 0, mg = 0;
  for (int r = 0; r < rows; ++r) {
    if (coast(pred, pk, false, thr, off, H, W, y0 + r, x)) mp |= 1ull << r;
    if (coast(target, tk, true, thr, off, H, W, y0 + r, x)) mg |= 1ull << r;
  }
  mask[((2 * b) * nb + blockIdx.y) * W + x] = mp;
  mask[((2 * b + 1) * nb + blockIdx.y) * W + x] = mg;
}

// ------------------------------------------------------------------------------------------------ pass 2: carries
// grid (ceil(W / 128), images): above[img][band][x] = last feature row in bands < band (-1 if none), below = first feature
// row in bands > band (INT_MAX if none).
__global__ void __launch_bounds__(COL_THREADS)
edt_carry_kernel(const unsigned long long* __restrict__ mask, int nb, int W, int* __restrict__ above,
                 int* __restrict__ below) {
  const int x = blockIdx.x * COL_THREADS + threadIdx.x;
  if (x >= W) return;
  const long long base = (long long)blockIdx.y * nb * W + x;
  int last = -1;
  for (int k = 0; k < nb; ++k) {
    above[base + (long long)k * W] = last;
    const unsigned long long m = mask[base + (long long)k * W];
    if (m) last = k * BAND + 63 - __clzll((long long)m);
  }
  int first = INT_MAX;
  for (int k = nb - 1; k >= 0; --k) {
    below[base + (long long)k * W] = first;
    const unsigned long long m = mask[base + (long long)k * W];
    if (m) first = k * BAND + __ffsll((long long)m) - 1;
  }
}

// ------------------------------------------------------------------------------------------------ pass 3: columns
// grid (ceil(W / 128), bands, images): g of 64 rows x 128 columns, transposed through shared memory into gT[img][x][Hp].
__global__ void __launch_bounds__(COL_THREADS)
edt_column_kernel(const unsigned long long* __restrict__ mask, const int* __restrict__ above,
                  const int* __restrict__ below, int H, int W, int Hp, uint16_t* __restrict__ gT) {
  constexpr int LDT = BAND + 2;                      // uint16 per tile row: 33 words, conflict-free column writes
  __shared__ __align__(16) uint16_t tile[COL_THREADS * LDT];
  const long long img = blockIdx.z, nb = gridDim.y;
  const int x0 = blockIdx.x * COL_THREADS, x = x0 + threadIdx.x;
  const int y0 = blockIdx.y * BAND;
  if (x < W) {
    const long long i = (img * nb + blockIdx.y) * W + x;
    const unsigned long long m = mask[i];
    const int a = above[i], bl = below[i];
    for (int r = 0; r < BAND; ++r) {
      const int y = y0 + r;
      int prev = a, next = bl;
      const unsigned long long lo = m & (r == 63 ? ~0ull : ((2ull << r) - 1));   // bits <= r
      if (lo) prev = y0 + 63 - __clzll((long long)lo);
      const unsigned long long hi = m >> r;                                       // bits >= r
      if (hi) next = y + __ffsll((long long)hi) - 1;
      int d = INT_MAX;
      if (prev >= 0) d = y - prev;
      if (next != INT_MAX) d = min(d, next - y);
      tile[threadIdx.x * LDT + r] = (y < H && d != INT_MAX) ? (uint16_t)d : NONE;
    }
  }
  __syncthreads();
  // 32 words per column: one warp stores one 128-byte column segment
  const uint32_t* t32 = reinterpret_cast<const uint32_t*>(tile);
  uint32_t* dst = reinterpret_cast<uint32_t*>(gT + img * W * (long long)Hp + y0);
  for (int e = threadIdx.x; e < COL_THREADS * (BAND / 2); e += COL_THREADS) {
    const int c = e >> 5, w = e & 31;
    if (x0 + c < W) dst[(long long)(x0 + c) * (Hp / 2) + w] = t32[c * (LDT / 2) + w];
  }
}

// ------------------------------------------------------------------------------------------------ pass 4: rows
__device__ __forceinline__ long long sq(long long v) { return v * v; }

// grid (Hp / 32, images), one warp: thread = row.  Stack entry q: stk = s | g << 16 (column, its g), stt = t (first column
// where the entry's parabola is the lowest).
__global__ void __launch_bounds__(32)
edt_row_kernel(const uint16_t* __restrict__ gT, int H, int W, int Hp, uint32_t* __restrict__ stk,
               uint16_t* __restrict__ stt, int* __restrict__ dist) {
  __shared__ int tile[32][33];
  const int lane = threadIdx.x;
  const long long img = blockIdx.y;
  const int y = blockIdx.x * 32 + lane;
  const long long col0 = img * W * (long long)Hp + y;          // element (x, y) of the [x][Hp] arrays is col0 + x * Hp
  const uint16_t* g = gT + col0;
  uint32_t* sk = stk + col0;
  uint16_t* sT = stt + col0;
  int q = -1, s = 0, gs = 0, t = 0;                            // stack depth - 1 and the top entry
  if (y < H) {
    for (int u0 = 0; u0 < W; u0 += 8) {
      uint16_t gv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) gv[j] = u0 + j < W ? __ldg(g + (long long)(u0 + j) * Hp) : NONE;
#pragma unroll 1
      for (int j = 0; j < 8; ++j) {
        if (gv[j] == NONE) continue;
        const int u = u0 + j, gu = gv[j];
        const long long fu = sq(gu);
        while (q >= 0 && sq(t - s) + sq(gs) > sq(t - u) + fu) {
          if (--q >= 0) {
            const uint32_t e = sk[(long long)q * Hp];
            s = e & 0xffff;
            gs = e >> 16;
            t = sT[(long long)q * Hp];
          }
        }
        int w = 0;
        if (q >= 0) {
          // Meijster's Sep: the last column where the top is not above the new parabola (the numerator is >= 0 here)
          w = 1 + (int)((sq(u) - sq(s) + fu - sq(gs)) / (2LL * (u - s)));
          if (w >= W) continue;
        }
        ++q;
        s = u;
        gs = gu;
        t = w;
        sk[(long long)q * Hp] = (uint32_t)s | ((uint32_t)gs << 16);
        sT[(long long)q * Hp] = (uint16_t)t;
      }
    }
  }
  int* out = dist + img * H * (long long)W;
  for (int c0 = (W - 1) & ~31; c0 >= 0; c0 -= 32) {
    for (int x = min(c0 + 31, W - 1); x >= c0; --x) {
      tile[lane][x - c0] = q < 0 ? -1 : (int)(sq(x - s) + sq(gs));
      if (q >= 0 && x == t && --q >= 0) {
        const uint32_t e = sk[(long long)q * Hp];
        s = e & 0xffff;
        gs = e >> 16;
        t = sT[(long long)q * Hp];
      }
    }
    __syncwarp();
    const int x = c0 + lane;
    for (int r = 0; r < 32; ++r) {
      const int yy = blockIdx.x * 32 + r;
      if (yy < H && x < W) out[(long long)yy * W + x] = tile[r][lane];
    }
    __syncwarp();
  }
}

int run_edt_passes(long long n, int H, int W, const Layout& L, uint8_t* ws, int* dist, cudaStream_t stream) {
  const int nb = (H + BAND - 1) / BAND, Hp = nb * BAND;
  auto* mask = reinterpret_cast<unsigned long long*>(ws + L.mask);
  int* above = reinterpret_cast<int*>(ws + L.above);
  int* below = reinterpret_cast<int*>(ws + L.below);
  auto* gT = reinterpret_cast<uint16_t*>(ws + L.gT);
  edt_carry_kernel<<<dim3(rbu_cdiv(W, COL_THREADS), (unsigned)n), COL_THREADS, 0, stream>>>(mask, nb, W, above, below);
  RBU_CHECK_LAUNCH();
  edt_column_kernel<<<dim3(rbu_cdiv(W, COL_THREADS), nb, (unsigned)n), COL_THREADS, 0, stream>>>(mask, above, below, H, W,
                                                                                                  Hp, gT);
  RBU_CHECK_LAUNCH();
  edt_row_kernel<<<dim3(Hp / 32, (unsigned)n), 32, 0, stream>>>(gT, H, W, Hp, reinterpret_cast<uint32_t*>(ws + L.stk),
                                                                reinterpret_cast<uint16_t*>(ws + L.stt), dist);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// ------------------------------------------------------------------------------------------------ coastline statistics
// Per (image b, direction dir): the samples are d2 = D[2b + 1 - dir] at the pixels of mask image 2b + dir (direction 0:
// D_G at the pixels of P; direction 1: D_P at the pixels of G).  d2 = -1 everywhere when the other coastline is empty.
//
// Order statistics: numpy's "linear" 95th percentile interpolates between ranks prev = floor((n - 1) * 0.95) and prev + 1
// (both n - 1 when that is past the end).  They are found with a four-level radix select over the 31-bit d2: level L
// counts byte 4 - L (bits 31-24, 23-16, 15-8, 7-0) of the samples whose higher bytes equal the prefix selected so far,
// per target rank (level 1 is shared by both).  Each level's blocks re-derive the prefixes from the earlier levels'
// histograms (a few 256-bin warp scans), so no separate select launch is needed.
struct Tol {
  int d2[MAX_T];
};

struct StatsWs {                   // per (b, dir): hist [4 levels][2 targets][256] u32, cnt [2 + MAX_T] u64, sums [tiles]
  unsigned* hist;
  unsigned long long* cnt;         // n, max d2 + 1 (0: none), tolerance counts
  double* sums;
  int tiles;
};

constexpr int HIST_WORDS = 4 * 2 * 256;
constexpr int CNT_WORDS = 2 + MAX_T;

// Warp 0: the bucket holding the need-th (1-based) element of a 256-bin histogram and the count before it.
__device__ __forceinline__ int select_byte(const unsigned* __restrict__ h, unsigned long long need,
                                           unsigned long long* before, unsigned long long* total) {
  const int lane = threadIdx.x & 31;
  unsigned v[8];
  unsigned long long sum = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i] = h[lane * 8 + i];
    sum += v[i];
  }
  unsigned long long incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  const unsigned long long excl = incl - sum;
  *total = __shfl_sync(0xffffffffu, incl, 31);
  const unsigned hit = __ballot_sync(0xffffffffu, excl < need && need <= incl);
  const int src = hit ? __ffs(hit) - 1 : 0;
  int bucket = 0;
  unsigned long long c = excl;
  if (lane == src) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (c + v[i] >= need) {
        bucket = lane * 8 + i;
        break;
      }
      c += v[i];
    }
  }
  *before = __shfl_sync(0xffffffffu, c, src);
  return __shfl_sync(0xffffffffu, bucket, src);
}

// Warp 0: ranks of the two order statistics from the valid sample count; false if there is none.
__device__ __forceinline__ bool pct_ranks(unsigned long long n, unsigned long long k[2]) {
  if (n == 0) return false;
  const double virt = (double)(n - 1) * 0.95;
  unsigned long long prev = (unsigned long long)floor(virt), next = prev + 1;
  if (virt >= (double)(n - 1)) prev = next = n - 1;
  k[0] = prev;
  k[1] = next;
  return true;
}

// Warp 0: for target j, the bytes selected by levels 1 .. levels (prefix) and the rank left inside that prefix.
__device__ __forceinline__ bool prefixes(const unsigned* __restrict__ hist, int levels, unsigned prefix[2],
                                         unsigned long long rank[2]) {
  unsigned long long before, total;
  select_byte(hist, 1, &before, &total);                    // the level-1 total = number of valid samples
  if (!pct_ranks(total, rank)) return false;
  for (int j = 0; j < 2; ++j) {
    unsigned p = 0;
    for (int l = 0; l < levels; ++l) {
      const int f = select_byte(hist + (l * 2 + (l ? j : 0)) * 256, rank[j] + 1, &before, &total);
      rank[j] -= before;
      p = (p << 8) | (unsigned)f;
    }
    prefix[j] = p;
  }
  return true;
}

// grid (tiles, 2, B), tile = 256 columns x 8 bands.  LEVEL 1 also reduces n, max, the tolerance counts and the per-tile
// float64 sum of sqrt(d2) (fixed order: bands, then bits, per thread; a fixed tree across the block).
template <int LEVEL>
__global__ void __launch_bounds__(ST_THREADS)
coast_stats_kernel(const unsigned long long* __restrict__ mask, const int* __restrict__ dist, int H, int W, int nb,
                   const __grid_constant__ Tol tol, int T, StatsWs sw) {
  __shared__ unsigned sh[2 * 256];
  __shared__ unsigned pre[2];
  __shared__ int live;
  __shared__ double red[ST_THREADS];
  const int b = blockIdx.z, dir = blockIdx.y;
  const long long sel = (long long)b * 2 + dir;
  unsigned* hist = sw.hist + sel * HIST_WORDS;
  for (int i = threadIdx.x; i < 2 * 256; i += ST_THREADS) sh[i] = 0;
  if (LEVEL > 1 && threadIdx.x < 32) {
    unsigned p[2];
    unsigned long long r[2];
    const bool ok = prefixes(hist, LEVEL - 1, p, r);
    if (threadIdx.x == 0) {
      live = ok;
      pre[0] = p[0];
      pre[1] = p[1];
    }
  }
  __syncthreads();
  if (LEVEL > 1 && !live) return;
  const int xt = (W + ST_THREADS - 1) / ST_THREADS;
  const int x = (blockIdx.x % xt) * ST_THREADS + threadIdx.x;
  const int k0 = (blockIdx.x / xt) * ST_BANDS;
  const long long src = 2LL * b + dir, other = 2LL * b + 1 - dir;
  const int* D = dist + other * H * (long long)W;
  constexpr int SHIFT = 32 - 8 * LEVEL;
  unsigned n = 0, within[MAX_T] = {};
  int mx = -1;
  double acc = 0.0;
  if (x < W) {
    for (int k = k0; k < min(k0 + ST_BANDS, nb); ++k) {
      unsigned long long m = mask[(src * nb + k) * W + x];
      while (m) {
        const int r = __ffsll((long long)m) - 1;
        m &= m - 1;
        const int d2 = __ldg(D + (long long)(k * BAND + r) * W + x);
        ++n;
        if (d2 < 0) continue;
        if constexpr (LEVEL == 1) {
          mx = max(mx, d2);
          acc += sqrt((double)d2);
#pragma unroll
          for (int t = 0; t < MAX_T; ++t) within[t] += (t < T && d2 <= tol.d2[t]);
          atomicAdd(&sh[d2 >> SHIFT], 1u);
        } else {
          const unsigned v = (unsigned)d2;
#pragma unroll
          for (int j = 0; j < 2; ++j)
            if ((v >> (SHIFT + 8)) == pre[j]) atomicAdd(&sh[j * 256 + ((v >> SHIFT) & 255u)], 1u);
        }
      }
    }
  }
  if (LEVEL == 1) {
    red[threadIdx.x] = acc;
    n = __reduce_add_sync(0xffffffffu, n);
    mx = __reduce_max_sync(0xffffffffu, mx);
#pragma unroll
    for (int t = 0; t < MAX_T; ++t) within[t] = __reduce_add_sync(0xffffffffu, within[t]);
    unsigned long long* cnt = sw.cnt + sel * CNT_WORDS;
    if ((threadIdx.x & 31) == 0) {
      if (n) atomicAdd(&cnt[0], (unsigned long long)n);
      if (mx >= 0) atomicMax(&cnt[1], (unsigned long long)mx + 1);
#pragma unroll
      for (int t = 0; t < MAX_T; ++t)
        if (within[t]) atomicAdd(&cnt[2 + t], (unsigned long long)within[t]);
    }
  }
  __syncthreads();
  if (LEVEL == 1) {
    for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
      if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) sw.sums[sel * sw.tiles + blockIdx.x] = red[0];
  }
  const int nbins = LEVEL == 1 ? 256 : 512;
  unsigned* dst = hist + (LEVEL - 1) * 512;
  for (int i = threadIdx.x; i < nbins; i += ST_THREADS)
    if (sh[i]) atomicAdd(&dst[i], sh[i]);
}

// grid (2, B), one block per (b, dir): the fixed-order sum of the tile sums, the two order statistics, stats_out.
__global__ void __launch_bounds__(ST_THREADS)
coast_final_kernel(StatsWs sw, int T, double* __restrict__ out) {
  __shared__ double red[ST_THREADS];
  __shared__ unsigned pre[2];
  __shared__ int live;
  const long long sel = (long long)blockIdx.y * 2 + blockIdx.x;
  const double* sums = sw.sums + sel * sw.tiles;
  double acc = 0.0;
  for (int i = threadIdx.x; i < sw.tiles; i += ST_THREADS) acc += sums[i];
  red[threadIdx.x] = acc;
  if (threadIdx.x < 32) {
    unsigned p[2];
    unsigned long long r[2];
    const bool ok = prefixes(sw.hist + sel * HIST_WORDS, 4, p, r);
    if (threadIdx.x == 0) {
      live = ok;
      pre[0] = p[0];
      pre[1] = p[1];
    }
  }
  __syncthreads();
  for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const unsigned long long* cnt = sw.cnt + sel * CNT_WORDS;
    double* o = out + sel * (5 + T);
    o[0] = (double)cnt[0];
    o[1] = live ? red[0] : -1.0;
    o[2] = live ? (double)(cnt[1] - 1) : -1.0;
    o[3] = live ? (double)pre[0] : -1.0;
    o[4] = live ? (double)pre[1] : -1.0;
    for (int t = 0; t < T; ++t) o[5 + t] = (double)cnt[2 + t];
  }
}

struct StatsLayout {
  Layout edt;
  size_t dist, hist, cnt, sums, total;
  int tiles;
};

StatsLayout stats_layout(int B, int H, int W) {
  StatsLayout S;
  S.edt = edt_layout(2LL * B, H, W);
  const int nb = (H + BAND - 1) / BAND;
  S.tiles = rbu_cdiv(W, ST_THREADS) * rbu_cdiv(nb, ST_BANDS);
  S.dist = S.edt.total;
  S.hist = align256(S.dist + (size_t)2 * B * H * W * 4);
  S.cnt = S.hist + (size_t)2 * B * HIST_WORDS * 4;             // hist and cnt are cleared together
  S.sums = align256(S.cnt + (size_t)2 * B * CNT_WORDS * 8);
  S.total = align256(S.sums + (size_t)2 * B * S.tiles * 8);
  return S;
}

bool dims_ok(int B, int H, int W) { return B > 0 && H >= 1 && W >= 1 && H <= 32768 && W <= 32768; }

}  // namespace

extern "C" size_t rbu_edt_workspace_bytes(int B, int H, int W) {
  if (!dims_ok(B, H, W) || B > 65535) return 0;
  return edt_layout(B, H, W).total;
}

extern "C" int rbu_edt(const uint8_t* features, int B, int H, int W, int32_t* dist2_out, void* workspace,
                       size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(features && dist2_out && workspace, "rbu_edt: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_edt: need B >= 1 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)", B, H, W);
  RBU_CHECK_ARG(B <= 65535, "rbu_edt: at most 65535 images per call");
  RBU_CHECK_ARG(workspace_bytes >= rbu_edt_workspace_bytes(B, H, W), "rbu_edt: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "rbu_edt: workspace must be 16-byte aligned");
  const Layout L = edt_layout(B, H, W);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const int nb = (H + BAND - 1) / BAND;
  edt_mask_kernel<<<dim3(rbu_cdiv(W, COL_THREADS), nb, B), COL_THREADS, 0, stream>>>(
      features, H, W, reinterpret_cast<unsigned long long*>(ws + L.mask));
  RBU_CHECK_LAUNCH();
  return run_edt_passes(B, H, W, L, ws, dist2_out, stream);
}

extern "C" size_t rbu_coastline_stats_workspace_bytes(int B, int H, int W) {
  if (!dims_ok(B, H, W) || B > 32767) return 0;
  return stats_layout(B, H, W).total;
}

extern "C" int rbu_coastline_stats(const void* pred, int pred_kind, const void* target, int target_kind, float threshold,
                                   int B, int H, int W, const int* tol_d2, int T, double* stats_out, void* workspace,
                                   size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(pred && target && stats_out && workspace, "rbu_coastline_stats: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_coastline_stats: need B >= 1 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)", B,
                H, W);
  RBU_CHECK_ARG(B <= 32767, "rbu_coastline_stats: at most 32767 images per call");
  RBU_CHECK_ARG((pred_kind == RBU_KIND_F32 || pred_kind == RBU_KIND_U8) &&
                    (target_kind == RBU_KIND_F32 || target_kind == RBU_KIND_U8),
                "rbu_coastline_stats: kinds must be RBU_KIND_F32 or RBU_KIND_U8");
  RBU_CHECK_ARG(T >= 0 && T <= MAX_T && (T == 0 || tol_d2), "rbu_coastline_stats: 0..%d tolerances", MAX_T);
  RBU_CHECK_ARG(workspace_bytes >= rbu_coastline_stats_workspace_bytes(B, H, W),
                "rbu_coastline_stats: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "rbu_coastline_stats: workspace must be 16-byte aligned");
  Tol tol;
  for (int t = 0; t < MAX_T; ++t) tol.d2[t] = t < T ? tol_d2[t] : -1;
  for (int t = 0; t < T; ++t) RBU_CHECK_ARG(tol.d2[t] >= 0, "rbu_coastline_stats: tolerance %d is negative", t);
  const StatsLayout S = stats_layout(B, H, W);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* dist = reinterpret_cast<int*>(ws + S.dist);
  auto* mask = reinterpret_cast<unsigned long long*>(ws + S.edt.mask);
  const int nb = (H + BAND - 1) / BAND;
  RBU_CHECK_CUDA(cudaMemsetAsync(ws + S.hist, 0, S.sums - S.hist, stream));
  coast_mask_kernel<<<dim3(rbu_cdiv(W, COL_THREADS), nb, B), COL_THREADS, 0, stream>>>(pred, pred_kind, target,
                                                                                       target_kind, threshold, H, W, mask);
  RBU_CHECK_LAUNCH();
  const int rc = run_edt_passes(2LL * B, H, W, S.edt, ws, dist, stream);
  if (rc != RBU_OK) return rc;
  StatsWs sw;
  sw.hist = reinterpret_cast<unsigned*>(ws + S.hist);
  sw.cnt = reinterpret_cast<unsigned long long*>(ws + S.cnt);
  sw.sums = reinterpret_cast<double*>(ws + S.sums);
  sw.tiles = S.tiles;
  const dim3 grid(S.tiles, 2, B);
  coast_stats_kernel<1><<<grid, ST_THREADS, 0, stream>>>(mask, dist, H, W, nb, tol, T, sw);
  RBU_CHECK_LAUNCH();
  coast_stats_kernel<2><<<grid, ST_THREADS, 0, stream>>>(mask, dist, H, W, nb, tol, T, sw);
  RBU_CHECK_LAUNCH();
  coast_stats_kernel<3><<<grid, ST_THREADS, 0, stream>>>(mask, dist, H, W, nb, tol, T, sw);
  RBU_CHECK_LAUNCH();
  coast_stats_kernel<4><<<grid, ST_THREADS, 0, stream>>>(mask, dist, H, W, nb, tol, T, sw);
  RBU_CHECK_LAUNCH();
  coast_final_kernel<<<dim3(2, B), ST_THREADS, 0, stream>>>(sw, T, stats_out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
