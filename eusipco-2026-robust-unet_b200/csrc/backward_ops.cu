// Bandwidth-bound backward kernels (K12 of SURVEY.md §2.1): the fused elementwise/reduction passes of
// ResidualBlock, AttentionGate, BatchNorm(+ReLU+Dropout2d), MaxPool and the `outc` head.
//
// Thread layout ("pattern B"): a block of 256 threads = rows x G, G = C/8 channel groups (power of two),
// each thread owns 8 channels of one pixel per iteration, so per-channel sums live in registers across the
// pixel loop and per-pixel sums are a reduction over the G threads of a row.  Grids are (chunks, N): one
// block covers a pixel chunk of ONE image, which makes per-(n,c) reductions local.  Partials are written
// per block and combined in a fixed order by a finalize kernel (deterministic, no float atomics).
#include "rbu_common.cuh"

namespace {

constexpr int NT = 256;

// sum over the G threads that share a pixel.  Contains __syncthreads() when G > 32: every thread of the
// block must call it the same number of times.
__device__ __forceinline__ float row_sum(float v, int G, float* red) {
  if (G <= 32) {
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  v = warp_sum(v);
  const int wpr = G >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  const int row = threadIdx.x / G;
  float t = 0.f;
  for (int i = 0; i < wpr; ++i) t += red[row * wpr + i];
  return t;
}

// reduce a per-thread 8-vector over the rows of the block and store it at dst[cg*8 .. +8]
__device__ __forceinline__ void rows_reduce_store(const float* acc, int G, int rows, float (*sv)[8], float* dst) {
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  __syncthreads();
#pragma unroll
  for (int e = 0; e < 8; ++e) sv[threadIdx.x][e] = acc[e];
  __syncthreads();
  if (row == 0) {
    float a[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] = sv[cg][e];
    for (int r = 1; r < rows; ++r)
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += sv[r * G + cg][e];
#pragma unroll
    for (int e = 0; e < 8; ++e) dst[cg * 8 + e] = a[e];
  }
}

// out[k] (+ optional out2) = sum over blocks of part[blk][k], fixed order, double accumulation
// Stage 1 of a long column reduction: slice s = blockIdx.y of the rows (rows s, s+S, ...) -> part2[s][K].  Rows of a
// slice are visited in order by 8 lanes with 4 independent loads in flight each; everything downstream sums the S
// slice rows in order, so the result is deterministic.
constexpr int COLSUM_SLICES = 32;
__global__ void __launch_bounds__(256)
colsum_stage1_kernel(const float* __restrict__ part, int nblk, int K, long blk_stride, float* __restrict__ part2) {
  __shared__ float sh[8][32];
  const int kx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + kx;
  const int S = gridDim.y, sl = blockIdx.y;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (k < K) {
    int b = sl + ly * S;
    const int step = 8 * S;
    for (; b + 3 * step < nblk; b += 4 * step) {
      a0 += part[(long)b * blk_stride + k];
      a1 += part[(long)(b + step) * blk_stride + k];
      a2 += part[(long)(b + 2 * step) * blk_stride + k];
      a3 += part[(long)(b + 3 * step) * blk_stride + k];
    }
    for (; b < nblk; b += step) a0 += part[(long)b * blk_stride + k];
  }
  sh[ly][kx] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (ly == 0 && k < K) {
    float t = 0.f;
    for (int j = 0; j < 8; ++j) t += sh[j][kx];
    part2[(long)sl * K + k] = t;
  }
}

// block = 32 columns x 8 lanes (launch with 256 threads, grid = ceil(K / 32))
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ part, int nblk, int K, long blk_stride, float* __restrict__ out, float post_scale) {
  __shared__ double sh[8][32];
  const int kx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + kx;
  double s = 0.0;
  if (k < K)
    for (int b = ly; b < nblk; b += 8) s += (double)part[(long)b * blk_stride + k];
  sh[ly][kx] = s;
  __syncthreads();
  if (ly == 0 && k < K) {
    double t = 0.0;
    for (int j = 0; j < 8; ++j) t += sh[j][kx];
    out[k] = (float)t * post_scale;
  }
}

// per-(n,c): out[n][c] = sum over the chunks of image n
__global__ void colsum_nc_kernel(const float* __restrict__ part, int N, int chunks, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (c >= C) return;
  double s = 0.0;
  for (int k = 0; k < chunks; ++k) s += (double)part[((long)n * chunks + k) * C + c];
  out[(long)n * C + c] = (float)s;
}

// ------------------------------------------------------------------------------------------------
// outc head backward (Main_Final.py:274-277): dz = dprobs * p (1-p); dx = dz * w; dw = sum dz x; db = sum dz
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT)
head_bwd_kernel(const float* __restrict__ dprobs, const float* __restrict__ probs, const bf16* __restrict__ x, long x_ld,
                bf16* __restrict__ dx, long dx_ld, long P, int C, const float* __restrict__ w, int px_per_block,
                float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const long p0 = (long)blockIdx.x * px_per_block;
  const long p1 = min(p0 + px_per_block, P);
  float wv[8], acc[8], accb[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { wv[e] = w[cg * 8 + e]; acc[e] = 0.f; accb[e] = 0.f; }
  if (row < rows) {
    for (long p = p0 + row; p < p1; p += rows) {
      const float pr = probs[p];
      const float dz = dprobs[p] * pr * (1.f - pr);
      float v[8], o[8];
      unpack8(ld_bf16x8_stream(x + p * x_ld + cg * 8), v);
#pragma unroll
      for (int e = 0; e < 8; ++e) { acc[e] += dz * v[e]; o[e] = dz * wv[e]; }
      if (cg == 0) accb[0] += dz;
      st_bf16x8(dx + p * dx_ld + cg * 8, pack8(o));
    }
  }
  __shared__ float sv[NT][8];
  float* dst = partials + (long)blockIdx.x * (C + 8);
  rows_reduce_store(acc, G, rows, sv, dst);
  __syncthreads();
  // bias partial: only cg == 0 threads carry it
#pragma unroll
  for (int e = 0; e < 8; ++e) sv[threadIdx.x][e] = accb[e];
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = 0.f;
    for (int r = 0; r < rows; ++r) b += sv[r * G][0];
    dst[C] = b;
  }
}

// ------------------------------------------------------------------------------------------------
// ResidualBlock backward (SURVEY.md Appendix C) in three passes over the activations:
//   pass 1  de = dout * [out > 0] (stored, may alias dout);  dG[p] = sum_c de * (A2g*y2 + B2g);
//           projection shortcut: per-channel sum(de), sum(de * ys)                       [-> SpatialAttention bwd]
//   pass 2  per (n,c):  D0 = sum_hw dc,  D1 = sum_hw dc * y2,
//           dc = de*gs + ds_avg/C + ds_max*[c == argmax_c]                               [-> rbu_rb_mid]
//   pass 3  dy2 = c1*dc + c0 + cy*y2 + cm*[pixel == argmax_hw];  dys = es*de + e0 + ey*ys
// Everything BatchNorm2 / ChannelAttention need between passes 2 and 3 (dT, the BN sums S1/S2, the gate MLP
// gradients) follows algebraically from D0/D1 and forward statistics, so no further pass over the data is needed.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT)
rb_bwd1_kernel(const bf16* __restrict__ dout, long dout_ld, const bf16* __restrict__ out, long out_ld,
               const bf16* __restrict__ y2, long y2_ld, bf16* __restrict__ de, long de_ld, const bf16* __restrict__ ys,
               long ys_ld, int HW, int C, int chunk_px, const float* __restrict__ A2g, const float* __restrict__ B2g,
               float* __restrict__ dG, float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_px, p1 = min(p0 + chunk_px, HW);
  constexpr int U = 2;
  const int iters = (p1 - p0 + rows * U - 1) / (rows * U);
  __shared__ float red[NT / 32];
  float a[8], b[8], acc1[8], acc2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    a[e] = A2g[(long)n * C + c];
    b[e] = B2g[(long)n * C + c];
    acc1[e] = 0.f;
    acc2[e] = 0.f;
  }
  for (int it = 0; it < iters; ++it) {
    bf16x8 rg[U], ro[U], ry[U], rs[U];
    bool act[U];
    // The four vectors of the NEXT iteration are prefetched into L2 while this one's are in flight (no registers held):
    // the kernel is latency-bound at two resident blocks per SM (ncu: 25 % warps active, 5 warps per issue on the long
    // scoreboard).  Same-box A/B, two alternations: 2.15 / 2.07 -> 1.93 / 1.97 ms per step.  The same prefetch made
    // rb_bwd3 (+3 %) and rb_bwd2 (+11 %) slower and left bn_bwd_apply / ag_bwd2 / ag_bwd3 unchanged, so only this kernel has it
    // (profiles/r02_i_ab_prefetch.txt).
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pl = p0 + ((it + 1) * U + u) * rows + row;
      if (row < rows && pl < p1) {
        const long p = (long)n * HW + pl;
        prefetch_l2(dout + p * dout_ld + cg * 8);
        prefetch_l2(out + p * out_ld + cg * 8);
        prefetch_l2(y2 + p * y2_ld + cg * 8);
        if (ys) prefetch_l2(ys + p * ys_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pl = p0 + (it * U + u) * rows + row;
      act[u] = row < rows && pl < p1;
      if (act[u]) {
        const long p = (long)n * HW + pl;
        rg[u] = ld_bf16x8_stream(dout + p * dout_ld + cg * 8);
        ro[u] = ld_bf16x8_stream(out + p * out_ld + cg * 8);
        ry[u] = ld_bf16x8(y2 + p * y2_ld + cg * 8);
        if (ys) rs[u] = ld_bf16x8(ys + p * ys_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pl = p0 + (it * U + u) * rows + row;
      const long p = (long)n * HW + pl;
      float part = 0.f;
      if (act[u]) {
        float g[8], o[8], y[8];
        unpack8(rg[u], g);
        unpack8(ro[u], o);
        unpack8(ry[u], y);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          g[e] = o[e] > 0.f ? g[e] : 0.f;
          part += g[e] * (a[e] * y[e] + b[e]);
        }
        st_bf16x8(de + p * de_ld + cg * 8, pack8(g));
        if (ys) {
          float sv8[8];
          unpack8(rs[u], sv8);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            acc1[e] += g[e];
            acc2[e] += g[e] * sv8[e];
          }
        }
      }
      part = row_sum(part, G, red);
      if (act[u] && cg == 0) dG[p] = part;
    }
  }
  if (ys) {
    __shared__ float sv[NT][8];
    float* dst = partials + ((long)n * gridDim.x + chunk) * 2 * C;
    rows_reduce_store(acc1, G, rows, sv, dst);
    rows_reduce_store(acc2, G, rows, sv, dst + C);
  }
}

// SpatialAttention backward (Main_Final.py:112-117), one shared-memory tiled kernel: dq = dG * gs (1-gs);
//   ds[k][h,w]   = sum_{r,q} K7[k][r][q] * dq[h-r+3, w-q+3]      (data gradient wrt [s_avg, s_max])
//   dK7[k][r][q] = sum_p dq[p] * s_k[p + (r-3, q-3)]             (98 per-thread accumulators, block partials)
// A block walks 32 x 16 tiles (grid-stride) holding the 38 x 22 halos of dq and s in shared memory; a thread owns four
// horizontally adjacent pixels, so one 10-wide window per halo row serves 4 x 7 taps (35 loads per pixel instead of 98).
constexpr int SB_TX = 32, SB_TY = 16, SB_HX = SB_TX + 6, SB_HY = SB_TY + 6, SB_NT = (SB_TX / 4) * SB_TY;
__global__ void __launch_bounds__(SB_NT)
sa_bwd_kernel(const float* __restrict__ dG, const float* __restrict__ gs, const float2* __restrict__ s, int N, int H, int W,
              const float* __restrict__ k7, float2* __restrict__ ds, float* __restrict__ partials) {
  __shared__ float wk[98];
  __shared__ float tq[SB_HY][SB_HX];
  __shared__ float2 tsv[SB_HY][SB_HX];
  const int tid = threadIdx.x;
  if (tid < 98) wk[tid] = k7[tid];
  float acc[98];
#pragma unroll
  for (int i = 0; i < 98; ++i) acc[i] = 0.f;
  const int tiles_x = (W + SB_TX - 1) / SB_TX, tiles_y = (H + SB_TY - 1) / SB_TY;
  const int tiles = tiles_x * tiles_y * N;
  const int tx = (tid % (SB_TX / 4)) * 4, ty = tid / (SB_TX / 4);
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int bx = t % tiles_x, by = (t / tiles_x) % tiles_y, n = t / (tiles_x * tiles_y);
    const int x0 = bx * SB_TX, y0 = by * SB_TY;
    const long nb = (long)n * H * W;
    __syncthreads();
    for (int i = tid; i < SB_HX * SB_HY; i += SB_NT) {
      const int hy = i / SB_HX, hx = i - hy * SB_HX;
      const int yy = y0 + hy - 3, xx = x0 + hx - 3;
      float q = 0.f;
      float2 sv = make_float2(0.f, 0.f);
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
        const long o = nb + (long)yy * W + xx;
        const float g = __ldg(&gs[o]);
        q = __ldg(&dG[o]) * g * (1.f - g);
        sv = __ldg(&s[o]);
      }
      tq[hy][hx] = q;
      tsv[hy][hx] = sv;
    }
    __syncthreads();
    const int x = x0 + tx, y = y0 + ty;
    if (x < W && y < H) {
      // dq of this thread's pixels (0 outside the image, so those pixels add nothing to the weight gradient)
      float dqc[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) dqc[e] = tq[ty + 3][tx + 3 + e];
      float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int r = 0; r < 7; ++r) {
        float2 sw[10];      // s at (y + r - 3, x + j - 3)
        float dw[10];       // dq at (y - r + 3, x + j - 3)
#pragma unroll
        for (int j = 0; j < 10; ++j) {
          sw[j] = tsv[ty + r][tx + j];
          dw[j] = tq[ty + 6 - r][tx + j];
        }
#pragma unroll
        for (int q = 0; q < 7; ++q) {
          const float w0 = wk[r * 7 + q], w1 = wk[49 + r * 7 + q];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            acc[r * 7 + q] += dqc[e] * sw[q + e].x;
            acc[49 + r * 7 + q] += dqc[e] * sw[q + e].y;
            const float dqq = dw[e + 6 - q];              // dq at (y - r + 3, x + e - q + 3)
            a0[e] += w0 * dqq;
            a1[e] += w1 * dqq;
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (x + e < W) ds[nb + (long)y * W + x + e] = make_float2(a0[e], a1[e]);
    }
  }
  __shared__ float sm[98][SB_NT / 32];
  const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int i = 0; i < 98; ++i) {
    const float v = warp_sum(acc[i]);
    if (lane == 0) sm[i][warp] = v;
  }
  __syncthreads();
  if (tid < 98) {
    float tsum = 0.f;
    for (int wq = 0; wq < SB_NT / 32; ++wq) tsum += sm[tid][wq];
    partials[(long)blockIdx.x * 98 + tid] = tsum;
  }
}

// pass 2: per-(n, chunk, c) partials of D0 = sum dc and D1 = sum dc * y2
__global__ void __launch_bounds__(NT)
rb_bwd2_kernel(const bf16* __restrict__ de, long de_ld, const bf16* __restrict__ y2, long y2_ld, int HW, int C,
               int chunk_px, const float* __restrict__ gs, const float2* __restrict__ ds, const int* __restrict__ amax_c,
               float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_px, p1 = min(p0 + chunk_px, HW);
  float acc0[8], acc1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { acc0[e] = 0.f; acc1[e] = 0.f; }
  const float invC = 1.f / (float)C;
  constexpr int U = 4;
  if (row < rows) {
    for (int pl0 = p0 + row; pl0 < p1; pl0 += rows * U) {
      bf16x8 rg[U], ry[U];
      float gsp[U];
      float2 d[U];
      int am[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int pl = pl0 + u * rows;
        if (pl < p1) {
          const long p = (long)n * HW + pl;
          rg[u] = ld_bf16x8_stream(de + p * de_ld + cg * 8);
          ry[u] = ld_bf16x8_stream(y2 + p * y2_ld + cg * 8);
          gsp[u] = __ldg(gs + p);
          d[u] = __ldg(ds + p);
          am[u] = __ldg(amax_c + p) - cg * 8;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (pl0 + u * rows < p1) {
          float g[8], y[8];
          unpack8(rg[u], g);
          unpack8(ry[u], y);
          const float base = d[u].x * invC;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float dc = g[e] * gsp[u] + base + (e == am[u] ? d[u].y : 0.f);
            acc0[e] += dc;
            acc1[e] += dc * y[e];
          }
        }
      }
    }
  }
  __shared__ float sv[NT][8];
  float* dst = partials + ((long)n * gridDim.x + chunk) * 2 * C;
  rows_reduce_store(acc0, G, rows, sv, dst);
  rows_reduce_store(acc1, G, rows, sv, dst + C);
}

// D[n][q][c] (double) = sum over the chunks of image n, chunk order
__global__ void rb_d_reduce_kernel(const float* __restrict__ part, int chunks, int C, double* __restrict__ D) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;   // over 2C
  const int n = blockIdx.y;
  if (k >= 2 * C) return;
  double s = 0.0;
  for (int j = 0; j < chunks; ++j) s += (double)part[((long)n * chunks + j) * 2 * C + k];
  D[(long)n * 2 * C + k] = s;
}

// pass 3 (streaming skeleton): dy2 = c1*dc + c0 + cy*y2 + cm*[pl == pstar];  dys = es*de + e0 + ey*ys
template <bool PROJ>
__global__ void __launch_bounds__(NT)
rb_bwd3_kernel(const bf16* __restrict__ de, long de_ld, const bf16* __restrict__ y2, long y2_ld, bf16* __restrict__ dy2,
               long dy2_ld, const bf16* __restrict__ ys, long ys_ld, bf16* __restrict__ dys, long dys_ld, int HW, int C,
               int lg, const float* __restrict__ gs, const float2* __restrict__ ds, const int* __restrict__ amax_c,
               const int* __restrict__ nc_arg, const float* __restrict__ c1, const float* __restrict__ c0,
               const float* __restrict__ cm, const float* __restrict__ cy, const float* __restrict__ es,
               const float* __restrict__ e0, const float* __restrict__ ey) {
  const int n = blockIdx.y, G = 1 << lg, items = HW << lg;
  const int cg = threadIdx.x & (G - 1);
  float k1[8], k0[8], km[8], ky[8];
  int pstar[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const long o = (long)n * C + cg * 8 + e;
    k1[e] = c1[o]; k0[e] = c0[o]; km[e] = cm[o]; ky[e] = cy[cg * 8 + e];
    pstar[e] = nc_arg[o];
  }
  float se[8], s0[8], sy[8];
  if (PROJ) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { se[e] = es[cg * 8 + e]; s0[e] = e0[cg * 8 + e]; sy[e] = ey[cg * 8 + e]; }
  }
  const float invC = 1.f / (float)C;
  const long ib = (long)n * HW;
  constexpr int U = 2;
  for (int base = blockIdx.x * (NT * U) + threadIdx.x; base < items; base += gridDim.x * (NT * U)) {
    bf16x8 rg[U], ry[U], rs[U];
    float gsp[U];
    float2 d[U];
    int am[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        const long p = ib + (i >> lg);
        rg[u] = ld_bf16x8_stream(de + p * de_ld + cg * 8);
        ry[u] = ld_bf16x8_stream(y2 + p * y2_ld + cg * 8);
        if (PROJ) rs[u] = ld_bf16x8_stream(ys + p * ys_ld + cg * 8);
        gsp[u] = __ldg(gs + p);
        d[u] = __ldg(ds + p);
        am[u] = __ldg(amax_c + p) - cg * 8;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        const int pl = i >> lg;
        const long p = ib + pl;
        float g[8], y[8], o[8];
        unpack8(rg[u], g);
        unpack8(ry[u], y);
        const float bse = d[u].x * invC;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float dc = g[e] * gsp[u] + bse + (e == am[u] ? d[u].y : 0.f);
          o[e] = k1[e] * dc + k0[e] + ky[e] * y[e] + (pl == pstar[e] ? km[e] : 0.f);
        }
        st_bf16x8(dy2 + p * dy2_ld + cg * 8, pack8(o));
        if (PROJ) {
          float sv8[8];
          unpack8(rs[u], sv8);
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = se[e] * g[e] + s0[e] + sy[e] * sv8[e];
          st_bf16x8(dys + p * dys_ld + cg * 8, pack8(o));
        }
      }
    }
  }
}

// ChannelAttention backward (Main_Final.py:97-101), one block per image
__global__ void __launch_bounds__(NT)
ca_bwd_n_kernel(const double* __restrict__ D, const float* __restrict__ scale2, const float* __restrict__ shift2,
                const float* __restrict__ g, const float* __restrict__ h_avg,
                const float* __restrict__ h_max, const float* __restrict__ V1, const float* __restrict__ V2, int C, int Ch,
                float* __restrict__ dt_out, float* __restrict__ dh_avg_out, float* __restrict__ dh_max_out,
                float* __restrict__ du_avg, float* __restrict__ du_max) {
  extern __shared__ float sm[];
  float* dt = sm;             // [C]
  float* dha = sm + C;        // [Ch]
  float* dhm = dha + Ch;      // [Ch]
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += NT) {
    const float gg = g[(long)n * C + c];
    // dT[n,c] = sum_hw dc * b,  b = scale2*y2 + shift2  ->  scale2*D1 + shift2*D0
    const float dT = (float)((double)scale2[c] * D[((long)n * 2 + 1) * C + c] + (double)shift2[c] * D[((long)n * 2 + 0) * C + c]);
    const float v = dT * gg * (1.f - gg);
    dt[c] = v;
    dt_out[(long)n * C + c] = v;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = warp; j < Ch; j += NT / 32) {
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a += V2[(long)c * Ch + j] * dt[c];
    a = warp_sum(a);
    if (lane == 0) {
      const float da = h_avg[(long)n * Ch + j] > 0.f ? a : 0.f;
      const float dm = h_max[(long)n * Ch + j] > 0.f ? a : 0.f;
      dha[j] = da;
      dhm[j] = dm;
      dh_avg_out[(long)n * Ch + j] = da;
      dh_max_out[(long)n * Ch + j] = dm;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += NT) {
    float a = 0.f, m = 0.f;
    for (int j = 0; j < Ch; ++j) {
      const float w = V1[(long)j * C + c];
      a += w * dha[j];
      m += w * dhm[j];
    }
    du_avg[(long)n * C + c] = a;
    du_max[(long)n * C + c] = m;
  }
}
// weight gradients of the shared MLP: block = 32 weights x 8 image lanes (lane j adds images j, j+8, ...; the lane sums
// are combined in lane order -> deterministic).  A thread per weight walking all N images was a 2 x 64-deep chain of
// dependent loads: 44 us per call for a few thousand values.
__global__ void __launch_bounds__(256)
ca_bwd_w_kernel(const float* __restrict__ dt, const float* __restrict__ dh_avg,
                const float* __restrict__ dh_max, const float* __restrict__ h_avg,
                const float* __restrict__ h_max, const float* __restrict__ u_avg,
                const float* __restrict__ u_max, int N, int C, int Ch, float* __restrict__ dV1,
                float* __restrict__ dV2) {
  __shared__ float sh[2][8][33];
  const int wx = threadIdx.x & 31, ln = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + wx;
  float s1 = 0.f, s2 = 0.f;
  if (i < C * Ch) {
    const int j1 = i / C, c1 = i - j1 * C;      // dV1[j][c]
    const int c2 = i / Ch, j2 = i - c2 * Ch;    // dV2[c][j]
    for (int n = ln; n < N; n += 8) {
      s1 += dh_avg[(long)n * Ch + j1] * u_avg[(long)n * C + c1] + dh_max[(long)n * Ch + j1] * u_max[(long)n * C + c1];
      s2 += dt[(long)n * C + c2] * (fmaxf(h_avg[(long)n * Ch + j2], 0.f) + fmaxf(h_max[(long)n * Ch + j2], 0.f));
    }
  }
  sh[0][ln][wx] = s1;
  sh[1][ln][wx] = s2;
  __syncthreads();
  if (ln == 0 && i < C * Ch) {
    float a = sh[0][0][wx], b = sh[1][0][wx];
    for (int r = 1; r < 8; ++r) { a += sh[0][r][wx]; b += sh[1][r][wx]; }
    dV1[i] = a;
    dV2[i] = b;
  }
}

// BatchNorm2 sums and the pass-3 coefficients, block = 32 channels x 8 lanes (lane j handles images j, j+8, ...;
// lane sums are combined in lane order -> deterministic):
//   S1[c] = sum_n (g*D0 + du_avg + du_max)
//   S2[c] = sum_n (g*rs*(D1 - mu*D0) + du_avg*(nc_mean - mu)*rs + du_max*(tv - mu)*rs)
//   c1 = scale2*g;  c0 = scale2*(du_avg/HW - S1/M + rs*mu*S2/M);  cy = -scale2*rs*S2/M;  cm = scale2*du_max
// and, for a projection shortcut with raw sums T1 = sum de, R = sum de*ys:
//   T2 = rs_s*(R - mu_s*T1);  es = scale_s;  e0 = scale_s*(-T1/M + rs_s*mu_s*T2/M);  ey = -scale_s*rs_s*T2/M
__global__ void __launch_bounds__(256)
rb_coef_kernel(const double* __restrict__ D, const float* __restrict__ g, const float* __restrict__ du_avg,
               const float* __restrict__ du_max, const float* __restrict__ nc_mean, const float* __restrict__ tv,
               const float* __restrict__ scale2, const float* __restrict__ mean2, const float* __restrict__ rstd2, int N,
               int HW, int C, float* __restrict__ sums2, float* __restrict__ c1, float* __restrict__ c0,
               float* __restrict__ cm, float* __restrict__ cy, const float* __restrict__ sraw /* [2C] or NULL */,
               const float* __restrict__ scale_s, const float* __restrict__ mean_s, const float* __restrict__ rstd_s,
               float* __restrict__ sums_s, float* __restrict__ es, float* __restrict__ e0, float* __restrict__ ey) {
  __shared__ double sh[2][8][32];
  __shared__ float bc[2][32];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  const bool ok = c < C;
  const double mu = ok ? (double)mean2[c] : 0.0, rs = ok ? (double)rstd2[c] : 0.0;
  double s1 = 0.0, s2 = 0.0;
  if (ok)
    for (int n = ly; n < N; n += 8) {
      const long o = (long)n * C + c;
      const double d0 = D[((long)n * 2 + 0) * C + c], d1 = D[((long)n * 2 + 1) * C + c];
      const double gg = g[o], da = du_avg[o], dm = du_max[o];
      s1 += gg * d0 + da + dm;
      s2 += gg * rs * (d1 - mu * d0) + da * ((double)nc_mean[o] - mu) * rs + dm * ((double)tv[o] - mu) * rs;
    }
  sh[0][ly][cx] = s1;
  sh[1][ly][cx] = s2;
  __syncthreads();
  const double M = (double)N * (double)HW;
  if (ly == 0 && ok) {
    double S1 = 0.0, S2 = 0.0;
    for (int j = 0; j < 8; ++j) { S1 += sh[0][j][cx]; S2 += sh[1][j][cx]; }
    sums2[c] = (float)S1;
    sums2[C + c] = (float)S2;
    bc[0][cx] = (float)(S1 / M);
    bc[1][cx] = (float)(S2 / M);
    cy[c] = (float)(-(double)scale2[c] * rs * S2 / M);
    if (sraw) {
      const double T1 = sraw[c], R = sraw[C + c], mus = mean_s[c], rss = rstd_s[c], scs = scale_s[c];
      const double T2 = rss * (R - mus * T1);
      sums_s[c] = (float)T1;
      sums_s[C + c] = (float)T2;
      es[c] = (float)scs;
      e0[c] = (float)(scs * (-T1 / M + rss * mus * T2 / M));
      ey[c] = (float)(-scs * rss * T2 / M);
    }
  }
  __syncthreads();
  if (ok) {
    const float s1m = bc[0][cx], s2m = bc[1][cx], sc = scale2[c];
    const float invHW = 1.f / (float)HW;
    for (int n = ly; n < N; n += 8) {
      const long o = (long)n * C + c;
      c1[o] = sc * g[o];
      c0[o] = sc * (du_avg[o] * invHW - s1m + (float)(rs * mu) * s2m);
      cm[o] = sc * du_max[o];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Generic BatchNorm(+ReLU)(+Dropout2d) backward: dz = dy * drop[n,c] * [scale*y+shift > 0]
//   reduce : per-channel A1 = sum dz, A2 = sum dz*y (raw y; the x-hat form follows in the finalize kernel)
//   final  : dbeta = A1, dgamma = rstd*(A2 - mean*A1); ky = -scale*rstd*dgamma/M, kc = -scale*A1/M - ky*mean
//   apply  : dx = scale*dz + kc + ky*y                                   (streaming skeleton)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT)
bn_bwd_reduce_kernel(const bf16* __restrict__ dy, long dy_ld, const bf16* __restrict__ y, long y_ld, int HW, int C,
                     int chunk_px, const float* __restrict__ scale, const float* __restrict__ shift,
                     const float* __restrict__ drop, int relu, float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_px, p1 = min(p0 + chunk_px, HW);
  float sc[8], sh[8], acc1[8], acc2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    sc[e] = scale[c]; sh[e] = shift[c];
    acc1[e] = 0.f; acc2[e] = 0.f;
  }
  constexpr int U = 4;
  if (row < rows) {
    for (int pl0 = p0 + row; pl0 < p1; pl0 += rows * U) {
      bf16x8 rg[U], rv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int pl = pl0 + u * rows;
        if (pl < p1) {
          const long p = (long)n * HW + pl;
          rg[u] = ld_bf16x8_stream(dy + p * dy_ld + cg * 8);
          rv[u] = ld_bf16x8_stream(y + p * y_ld + cg * 8);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (pl0 + u * rows < p1) {
          float g[8], v[8];
          unpack8(rg[u], g);
          unpack8(rv[u], v);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float dz = (relu && !(sc[e] * v[e] + sh[e] > 0.f)) ? 0.f : g[e];
            acc1[e] += dz;
            acc2[e] += dz * v[e];
          }
        }
      }
    }
  }
  // Dropout2d scale is constant per (n,c): apply it once per block instead of per element
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float d = drop ? drop[(long)n * C + cg * 8 + e] : 1.f;
    acc1[e] *= d;
    acc2[e] *= d;
  }
  __shared__ float sv[NT][8];
  float* dst = partials + ((long)n * gridDim.x + chunk) * 2 * C;
  rows_reduce_store(acc1, G, rows, sv, dst);
  rows_reduce_store(acc2, G, rows, sv, dst + C);
}

// block = 32 channels x 8 lanes over the nblk partial rows (fixed order); writes sums[2C] and coef[2C] = (kc, ky)
__global__ void __launch_bounds__(256)
bn_bwd_final_kernel(const float* __restrict__ part, int nblk, int C, const float* __restrict__ scale,
                    const float* __restrict__ mean, const float* __restrict__ rstd, float invM, float* __restrict__ sums,
                    float* __restrict__ coef) {
  __shared__ double sh[2][8][32];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  double a1 = 0.0, a2 = 0.0;
  if (c < C)
    for (int b = ly; b < nblk; b += 8) {
      a1 += (double)part[(long)b * 2 * C + c];
      a2 += (double)part[(long)b * 2 * C + C + c];
    }
  sh[0][ly][cx] = a1;
  sh[1][ly][cx] = a2;
  __syncthreads();
  if (ly == 0 && c < C) {
    double A1 = 0.0, A2 = 0.0;
    for (int j = 0; j < 8; ++j) { A1 += sh[0][j][cx]; A2 += sh[1][j][cx]; }
    const double mu = mean[c], rs = rstd[c], sc = scale[c];
    const double dgamma = rs * (A2 - mu * A1);
    sums[c] = (float)A1;
    sums[C + c] = (float)dgamma;
    const double ky = -sc * rs * dgamma * (double)invM;
    coef[c] = (float)(-sc * A1 * (double)invM - ky * mu);
    coef[C + c] = (float)ky;
  }
}

__global__ void __launch_bounds__(NT)
bn_bwd_apply_kernel(const bf16* __restrict__ dy, long dy_ld, const bf16* __restrict__ y, long y_ld, bf16* __restrict__ dx,
                    long dx_ld, int HW, int C, int lg, const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ drop, int relu, const float* __restrict__ coef) {
  const int n = blockIdx.y, G = 1 << lg, items = HW << lg;
  const int cg = threadIdx.x & (G - 1);
  float sc[8], sh[8], sd[8], kc[8], ky[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    sc[e] = scale[c]; sh[e] = shift[c];
    sd[e] = sc[e] * (drop ? drop[(long)n * C + c] : 1.f);
    kc[e] = coef[c]; ky[e] = coef[C + c];
  }
  const long ib = (long)n * HW;
  constexpr int U = 4;
  for (int base = blockIdx.x * (NT * U) + threadIdx.x; base < items; base += gridDim.x * (NT * U)) {
    bf16x8 rg[U], rv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        const long p = ib + (i >> lg);
        rg[u] = ld_bf16x8_stream(dy + p * dy_ld + cg * 8);
        rv[u] = ld_bf16x8_stream(y + p * y_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        float g[8], v[8];
        unpack8(rg[u], g);
        unpack8(rv[u], v);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float dz = (relu && !(sc[e] * v[e] + sh[e] > 0.f)) ? 0.f : g[e];
          g[e] = sd[e] * dz + kc[e] + ky[e] * v[e];
        }
        st_bf16x8(dx + (ib + (i >> lg)) * dx_ld + cg * 8, pack8(g));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// AttentionGate backward (Main_Final.py:143-148)
// pass 1 (over C): dskip = da * psi; dpsi = sum_c da * skip; dq = dpsi psi (1-psi) -> dq[P];
//                  block partials: sum(dq), sum(dq * qhat)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT)
ag_bwd1_kernel(const bf16* __restrict__ da, long da_ld, const bf16* __restrict__ skip, long s_ld, bf16* __restrict__ dskip,
               long ds_ld, int HW, int C, int chunk_px, const float* __restrict__ psi, const float* __restrict__ q0,
               const float* __restrict__ stats, float* __restrict__ dq_out, float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_px, p1 = min(p0 + chunk_px, HW);
  constexpr int U = 2;
  const int iters = (p1 - p0 + rows * U - 1) / (rows * U);
  __shared__ float red[NT / 32];
  const float mean = stats[2], rstd = stats[3];
  float l0 = 0.f, l1 = 0.f;
  for (int it = 0; it < iters; ++it) {
    bf16x8 rg[U], rx[U];
    float ps[U];
    bool act[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pl = p0 + (it * U + u) * rows + row;
      act[u] = row < rows && pl < p1;
      if (act[u]) {
        const long p = (long)n * HW + pl;
        rg[u] = ld_bf16x8_stream(da + p * da_ld + cg * 8);
        rx[u] = ld_bf16x8(skip + p * s_ld + cg * 8);
        ps[u] = __ldg(psi + p);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pl = p0 + (it * U + u) * rows + row;
      const long p = (long)n * HW + pl;
      float part = 0.f;
      if (act[u]) {
        float g[8], x[8];
        unpack8(rg[u], g);
        unpack8(rx[u], x);
#pragma unroll
        for (int e = 0; e < 8; ++e) { part += g[e] * x[e]; g[e] *= ps[u]; }
        st_bf16x8(dskip + p * ds_ld + cg * 8, pack8(g));
      }
      part = row_sum(part, G, red);
      if (act[u] && cg == 0) {
        const float dq = part * ps[u] * (1.f - ps[u]);
        dq_out[p] = dq;
        l0 += dq;
        l1 += dq * (q0[p] - mean) * rstd;
      }
    }
  }
  __shared__ float r0[NT / 32], r1[NT / 32];
  l0 = warp_sum(l0);
  l1 = warp_sum(l1);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { r0[threadIdx.x >> 5] = l0; r1[threadIdx.x >> 5] = l1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int w = 0; w < NT / 32; ++w) { a += r0[w]; b += r1[w]; }
    float* dst = partials + ((long)n * gridDim.x + chunk) * 2;
    dst[0] = a;
    dst[1] = b;
  }
}

// pass 2 (over F), reduce: dq0 = a_psi*(dq - c1 - qhat*c2); t = Ag yg + Ax yx + (Bg+Bx); dt = wpsi*dq0*[t>0]
//   per-channel sums: relu(t)*dq0 [dwpsi], dt, dt*yg, dt*yx (raw; x-hat forms follow in the finalize kernel)
__global__ void __launch_bounds__(NT)
ag_bwd2_kernel(const bf16* __restrict__ yg, long yg_ld, const bf16* __restrict__ yx, long yx_ld, int HW, int F,
               int chunk_px, const float* __restrict__ Ag, const float* __restrict__ Bg, const float* __restrict__ Ax,
               const float* __restrict__ Bx, const float* __restrict__ wpsi, const float* __restrict__ dq,
               const float* __restrict__ q0, const float* __restrict__ stats,
               const float* __restrict__ csum /* [2]: sum(dq), sum(dq*qhat) */, float invM, float* __restrict__ partials) {
  const int G = F >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_px, p1 = min(p0 + chunk_px, HW);
  const float a_psi = stats[0], mean = stats[2], rstd = stats[3];
  const float c1 = csum[0] * invM, c2 = csum[1] * invM;
  float ag[8], ax[8], bs[8], wp[8], acc[4][8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    ag[e] = Ag[c]; ax[e] = Ax[c]; bs[e] = Bg[c] + Bx[c]; wp[e] = wpsi[c];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q][e] = 0.f;
  }
  constexpr int U = 2;
  if (row < rows) {
    for (int pl0 = p0 + row; pl0 < p1; pl0 += rows * U) {
      bf16x8 ra[U], rb[U];
      float dqv[U], qv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int pl = pl0 + u * rows;
        if (pl < p1) {
          const long p = (long)n * HW + pl;
          ra[u] = ld_bf16x8_stream(yg + p * yg_ld + cg * 8);
          rb[u] = ld_bf16x8_stream(yx + p * yx_ld + cg * 8);
          dqv[u] = __ldg(dq + p);
          qv[u] = __ldg(q0 + p);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (pl0 + u * rows < p1) {
          float a[8], b[8];
          unpack8(ra[u], a);
          unpack8(rb[u], b);
          const float dq0 = a_psi * (dqv[u] - c1 - (qv[u] - mean) * rstd * c2);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float t = ag[e] * a[e] + ax[e] * b[e] + bs[e];
            const float dt = t > 0.f ? wp[e] * dq0 : 0.f;
            acc[0][e] += fmaxf(t, 0.f) * dq0;
            acc[1][e] += dt;
            acc[2][e] += dt * a[e];
            acc[3][e] += dt * b[e];
          }
        }
      }
    }
  }
  __shared__ float sv[NT][8];
  float* dst = partials + ((long)n * gridDim.x + chunk) * 4 * F;
#pragma unroll
  for (int q = 0; q < 4; ++q) rows_reduce_store(acc[q], G, rows, sv, dst + q * F);
}

// sums_f[4][F] = dwpsi, dbeta (shared by W_g.1 / W_x.1), dgamma_g, dgamma_x; coef[4][F] = kgc, kgy, kxc, kxy with
// dyg = Ag*dt + kgc + kgy*yg and dyx = Ax*dt + kxc + kxy*yx
__global__ void __launch_bounds__(256)
ag_bwd_final_kernel(const float* __restrict__ part, int nblk, int F, const float* __restrict__ Ag,
                    const float* __restrict__ Ax, const float* __restrict__ mg, const float* __restrict__ rg,
                    const float* __restrict__ mx, const float* __restrict__ rx, float invM, float* __restrict__ sums_f,
                    float* __restrict__ coef) {
  __shared__ double sh[4][8][32];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  double a[4] = {0.0, 0.0, 0.0, 0.0};
  if (c < F)
    for (int b = ly; b < nblk; b += 8)
#pragma unroll
      for (int q = 0; q < 4; ++q) a[q] += (double)part[(long)b * 4 * F + q * F + c];
#pragma unroll
  for (int q = 0; q < 4; ++q) sh[q][ly][cx] = a[q];
  __syncthreads();
  if (ly == 0 && c < F) {
    double A[4] = {0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) A[q] += sh[q][j][cx];
    const double dgg = (double)rg[c] * (A[2] - (double)mg[c] * A[1]);
    const double dgx = (double)rx[c] * (A[3] - (double)mx[c] * A[1]);
    sums_f[c] = (float)A[0];
    sums_f[F + c] = (float)A[1];
    sums_f[2 * F + c] = (float)dgg;
    sums_f[3 * F + c] = (float)dgx;
    const double kgy = -(double)Ag[c] * rg[c] * dgg * invM, kxy = -(double)Ax[c] * rx[c] * dgx * invM;
    coef[c] = (float)(-(double)Ag[c] * A[1] * invM - kgy * mg[c]);
    coef[F + c] = (float)kgy;
    coef[2 * F + c] = (float)(-(double)Ax[c] * A[1] * invM - kxy * mx[c]);
    coef[3 * F + c] = (float)kxy;
  }
}

// pass 3 (over F), streaming skeleton: dyg, dyx
__global__ void __launch_bounds__(NT)
ag_bwd3_kernel(const bf16* __restrict__ yg, long yg_ld, const bf16* __restrict__ yx, long yx_ld, bf16* __restrict__ dyg,
               long dyg_ld, bf16* __restrict__ dyx, long dyx_ld, int HW, int F, int lg, const float* __restrict__ Ag,
               const float* __restrict__ Bg, const float* __restrict__ Ax, const float* __restrict__ Bx,
               const float* __restrict__ wpsi, const float* __restrict__ dq, const float* __restrict__ q0,
               const float* __restrict__ stats, const float* __restrict__ csum, float invM,
               const float* __restrict__ coef) {
  const int n = blockIdx.y, G = 1 << lg, items = HW << lg;
  const int cg = threadIdx.x & (G - 1);
  const float a_psi = stats[0], mean = stats[2], rstd = stats[3];
  const float c1 = csum[0] * invM, c2 = csum[1] * invM;
  float ag[8], ax[8], bs[8], agw[8], axw[8], kgc[8], kgy[8], kxc[8], kxy[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    ag[e] = Ag[c]; ax[e] = Ax[c]; bs[e] = Bg[c] + Bx[c];
    agw[e] = ag[e] * wpsi[c]; axw[e] = ax[e] * wpsi[c];
    kgc[e] = coef[c]; kgy[e] = coef[F + c]; kxc[e] = coef[2 * F + c]; kxy[e] = coef[3 * F + c];
  }
  const long ib = (long)n * HW;
  constexpr int U = 2;
  for (int base = blockIdx.x * (NT * U) + threadIdx.x; base < items; base += gridDim.x * (NT * U)) {
    bf16x8 ra[U], rb[U];
    float dqv[U], qv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        const long p = ib + (i >> lg);
        ra[u] = ld_bf16x8_stream(yg + p * yg_ld + cg * 8);
        rb[u] = ld_bf16x8_stream(yx + p * yx_ld + cg * 8);
        dqv[u] = __ldg(dq + p);
        qv[u] = __ldg(q0 + p);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = base + u * NT;
      if (i < items) {
        const long p = ib + (i >> lg);
        float a[8], b[8], og[8], ox[8];
        unpack8(ra[u], a);
        unpack8(rb[u], b);
        const float dq0 = a_psi * (dqv[u] - c1 - (qv[u] - mean) * rstd * c2);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float t = ag[e] * a[e] + ax[e] * b[e] + bs[e];
          const float m = t > 0.f ? dq0 : 0.f;
          og[e] = agw[e] * m + kgc[e] + kgy[e] * a[e];
          ox[e] = axw[e] * m + kxc[e] + kxy[e] * b[e];
        }
        st_bf16x8(dyg + p * dyg_ld + cg * 8, pack8(og));
        st_bf16x8(dyx + p * dyx_ld + cg * 8, pack8(ox));
      }
    }
  }
}

// 2x2 max-pool backward: route dy to the FIRST maximal input in scan order and ADD it to dx
__global__ void __launch_bounds__(NT)
maxpool_bwd_kernel(const bf16* __restrict__ x, long x_ld, const bf16* __restrict__ dy, long dy_ld, bf16* __restrict__ dx,
                   long dx_ld, int N, int Ho, int Wo, int C, int accumulate) {
  const int G = C >> 3;
  const long total = (long)N * Ho * Wo * G;
  const int W = 2 * Wo;
  for (long i = blockIdx.x * (long)NT + threadIdx.x; i < total; i += (long)gridDim.x * NT) {
    const int cg = (int)(i % G);
    const long po = i / G;
    const int wo = (int)(po % Wo);
    const int ho = (int)((po / Wo) % Ho);
    const int n = (int)(po / ((long)Wo * Ho));
    const long pi = ((long)n * 2 * Ho + 2 * ho) * W + 2 * wo;
    const long off[4] = {pi, pi + 1, pi + W, pi + W + 1};
    float v[4][8], g[8], o[4][8];
    unpack8(ld_bf16x8_stream(dy + po * dy_ld + cg * 8), g);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      unpack8(ld_bf16x8(x + off[q] * x_ld + cg * 8), v[q]);
      if (accumulate) unpack8(ld_bf16x8(dx + off[q] * dx_ld + cg * 8), o[q]);
      else {
#pragma unroll
        for (int e = 0; e < 8; ++e) o[q][e] = 0.f;
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int best = 0;
      float bv = v[0][e];
#pragma unroll
      for (int q = 1; q < 4; ++q)
        if (v[q][e] > bv) { bv = v[q][e]; best = q; }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q == best) o[q][e] += g[e];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) st_bf16x8(dx + off[q] * dx_ld + cg * 8, pack8(o[q]));
  }
}

// per-channel sum over pixels of a bf16 view (bias gradients)
__global__ void __launch_bounds__(NT)
chan_sum_kernel(const bf16* __restrict__ x, long ld, long P, int C, int px_per_block, float* __restrict__ partials) {
  const int G = C >> 3, rows = NT / G;
  const int cg = threadIdx.x % G, row = threadIdx.x / G;
  const long p0 = (long)blockIdx.x * px_per_block;
  const long p1 = min(p0 + px_per_block, P);
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  if (row < rows)
    for (long p = p0 + row; p < p1; p += rows) {
      float v[8];
      unpack8(ld_bf16x8_stream(x + p * ld + cg * 8), v);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
  __shared__ float sv[NT][8];
  rows_reduce_store(acc, G, rows, sv, partials + (long)blockIdx.x * C);
}

// ---------------------------------------------------------------------------------- host helpers
bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

int bwd_chunks(int N, int HW, int C) {
  const int rows = NT / (C >> 3);
  long want = ((long)rbu_num_sms() * 16 + N - 1) / N;    // ~16 blocks per SM in total: small tail wave
  long maxc = (HW + (long)rows * 4 - 1) / ((long)rows * 4);
  if (maxc < 1) maxc = 1;
  if (want > maxc) want = maxc;
  if (want < 1) want = 1;
  return (int)want;
}

int flat_blocks(long P, int C, int* px_per_block) {
  const int rows = NT / (C >> 3);
  long blocks = (long)rbu_num_sms() * 16;
  long maxb = (P + (long)rows * 4 - 1) / ((long)rows * 4);
  if (maxb < 1) maxb = 1;
  if (blocks > maxb) blocks = maxb;
  *px_per_block = (int)((P + blocks - 1) / blocks);
  return (int)((P + *px_per_block - 1) / *px_per_block);
}

int grid1d(long items, int per_block) {
  long b = (items + per_block - 1) / per_block;
  const long cap = (long)rbu_num_sms() * 8;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// Long partial lists ([nblk][stride] rows) are first folded into COLSUM_SLICES rows of K columns in `scratch`
// (which must hold COLSUM_SLICES*K floats); short ones are passed through.  Updates part / nblk / stride in place.
int colsum_fold(const float*& part, int& nblk, long& stride, int K, float* scratch, cudaStream_t st) {
  if (nblk <= 4 * COLSUM_SLICES) return RBU_OK;
  colsum_stage1_kernel<<<dim3(rbu_cdiv(K, 32), COLSUM_SLICES), 256, 0, st>>>(part, nblk, K, stride, scratch);
  RBU_CHECK_LAUNCH();
  part = scratch;
  nblk = COLSUM_SLICES;
  stride = K;
  return RBU_OK;
}

}  // namespace

#define VIEW_OK(ptr, ld) ((ptr) != nullptr && ((uintptr_t)(ptr) & 15) == 0 && (ld) % 8 == 0)
#define CH_OK(C) ((C) >= 8 && (C) <= 2048 && pow2(C))
#define FOLD_FLOATS(K) ((size_t)COLSUM_SLICES * (K))

size_t colsum_scratch_floats(int K) { return FOLD_FLOATS(K); }

int colsum_split(const float* part, int nblk, long stride, int K1, float* out1, int K2, float* out2, float* scratch,
                 cudaStream_t st) {
  int rc = colsum_fold(part, nblk, stride, K1 + K2, scratch, st);
  if (rc) return rc;
  colsum_kernel<<<rbu_cdiv(K1, 32), 256, 0, st>>>(part, nblk, K1, stride, out1, 1.f);
  RBU_CHECK_LAUNCH();
  colsum_kernel<<<rbu_cdiv(K2, 32), 256, 0, st>>>(part + K1, nblk, K2, stride, out2, 1.f);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// Workspace (floats) large enough for every backward pass of a [N,HW,C] tensor: max partial layout is
// [N*chunks][4][C] (AttentionGate pass 2); the head / chan_sum layouts are smaller.
extern "C" size_t rbu_bwd_workspace_bytes(int N, int HW, int C) {
  if (!CH_OK(C)) return 0;
  int ppb;
  const size_t a = (size_t)N * bwd_chunks(N, HW, C) * 4 * C + 4 * C + FOLD_FLOATS(4 * C + 128);
  const size_t b = (size_t)flat_blocks((long)N * HW, C, &ppb) * (C + 8) + FOLD_FLOATS(C + 8);
  const size_t c = (size_t)rbu_num_sms() * 8 * 98 + FOLD_FLOATS(128);
  size_t m = a > b ? a : b;
  if (c > m) m = c;
  return m * sizeof(float);
}

extern "C" int rbu_head_backward(const float* dprobs, const float* probs, const void* x, int64_t x_ld, void* dx,
                                 int64_t dx_ld, int64_t P, int C, const float* w, float* dw, float* db, void* workspace,
                                 size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(dprobs && probs && VIEW_OK(x, x_ld) && VIEW_OK(dx, dx_ld) && w && dw && db && CH_OK(C) && C <= 256,
                "rbu_head_backward: bad arguments");
  int ppb;
  const int blocks = flat_blocks(P, C, &ppb);
  RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)blocks * (C + 8) * sizeof(float), "rbu_head_backward: workspace too small");
  float* part = (float*)workspace;
  head_bwd_kernel<<<blocks, NT, 0, st>>>(dprobs, probs, (const bf16*)x, x_ld, (bf16*)dx, dx_ld, P, C, w, ppb, part);
  RBU_CHECK_LAUNCH();
  const float* pp = part;
  int nb2 = blocks;
  long stride = C + 8;
  RBU_CHECK_ARG(workspace_bytes >= ((size_t)blocks * (C + 8) + FOLD_FLOATS(C + 8)) * sizeof(float), "rbu_head_backward: workspace too small");
  int rc = colsum_fold(pp, nb2, stride, C + 1, part + (size_t)blocks * (C + 8), st);
  if (rc) return rc;
  colsum_kernel<<<rbu_cdiv(C, 32), 256, 0, st>>>(pp, nb2, C, stride, dw, 1.f);
  RBU_CHECK_LAUNCH();
  colsum_kernel<<<1, 256, 0, st>>>(pp + C, nb2, 1, stride, db, 1.f);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_rb_bwd1(const void* dout, int64_t dout_ld, const void* out, int64_t out_ld, const void* y2,
                           int64_t y2_ld, void* de, int64_t de_ld, const void* ys, int64_t ys_ld, int N, int HW, int C,
                           const float* A2g, const float* B2g, float* dG, float* sums_s_raw, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(dout, dout_ld) && VIEW_OK(out, out_ld) && VIEW_OK(y2, y2_ld) && VIEW_OK(de, de_ld) && A2g && B2g &&
                    dG && CH_OK(C) && N > 0 && N <= 65535 && HW > 0, "rbu_rb_bwd1: bad arguments");
  RBU_CHECK_ARG(!ys || (VIEW_OK(ys, ys_ld) && sums_s_raw), "rbu_rb_bwd1: projection-shortcut arguments missing");
  const int chunks = bwd_chunks(N, HW, C);
  RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)N * chunks * 2 * C * sizeof(float), "rbu_rb_bwd1: workspace too small");
  rb_bwd1_kernel<<<dim3(chunks, N), NT, 0, st>>>((const bf16*)dout, dout_ld, (const bf16*)out, out_ld, (const bf16*)y2,
                                                 y2_ld, (bf16*)de, de_ld, (const bf16*)ys, ys_ld, HW, C,
                                                 rbu_cdiv(HW, chunks), A2g, B2g, dG, (float*)workspace);
  RBU_CHECK_LAUNCH();
  if (ys) {
    const float* pp = (const float*)workspace;
    int nb2 = N * chunks;
    long stride = 2 * C;
    RBU_CHECK_ARG(workspace_bytes >= ((size_t)N * chunks * 2 * C + FOLD_FLOATS(2 * C)) * sizeof(float), "rbu_rb_bwd1: workspace too small");
    int rc = colsum_fold(pp, nb2, stride, 2 * C, (float*)workspace + (size_t)N * chunks * 2 * C, st);
    if (rc) return rc;
    colsum_kernel<<<rbu_cdiv(2 * C, 32), 256, 0, st>>>(pp, nb2, 2 * C, stride, sums_s_raw, 1.f);
    RBU_CHECK_LAUNCH();
  }
  return RBU_OK;
}

extern "C" int rbu_sa_bwd(const float* dG, const float* gs, const float* s, int N, int H, int W, const float* k7,
                          float* ds, float* dk7, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(dG && gs && s && k7 && ds && dk7 && N > 0 && H > 0 && W > 0, "rbu_sa_bwd: bad arguments");
  const long tiles = (long)rbu_cdiv(W, SB_TX) * rbu_cdiv(H, SB_TY) * N;
  const long cap = (long)rbu_num_sms() * 6;
  const int blocks = (int)(tiles < cap ? tiles : cap);
  RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)blocks * 98 * sizeof(float), "rbu_sa_bwd: workspace too small");
  sa_bwd_kernel<<<blocks, SB_NT, 0, st>>>(dG, gs, (const float2*)s, N, H, W, k7, (float2*)ds, (float*)workspace);
  RBU_CHECK_LAUNCH();
  const float* pp = (const float*)workspace;
  int nb2 = blocks;
  long stride = 98;
  RBU_CHECK_ARG(workspace_bytes >= ((size_t)blocks * 98 + FOLD_FLOATS(98)) * sizeof(float), "rbu_sa_bwd: workspace too small");
  int rc = colsum_fold(pp, nb2, stride, 98, (float*)workspace + (size_t)blocks * 98, st);
  if (rc) return rc;
  colsum_kernel<<<rbu_cdiv(98, 32), 256, 0, st>>>(pp, nb2, 98, stride, dk7, 1.f);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// pass 2: D[N][2][C] (double) = per-(n,c) sum dc, sum dc*y2
extern "C" int rbu_rb_bwd2(const void* de, int64_t de_ld, const void* y2, int64_t y2_ld, int N, int HW, int C,
                           const float* gs, const float* ds, const int* amax_c, double* D, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(de, de_ld) && VIEW_OK(y2, y2_ld) && CH_OK(C) && N > 0 && N <= 65535 && HW > 0 && gs && ds && amax_c && D,
                "rbu_rb_bwd2: bad arguments");
  const int chunks = bwd_chunks(N, HW, C);
  RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)N * chunks * 2 * C * sizeof(float), "rbu_rb_bwd2: workspace too small");
  rb_bwd2_kernel<<<dim3(chunks, N), NT, 0, st>>>((const bf16*)de, de_ld, (const bf16*)y2, y2_ld, HW, C, rbu_cdiv(HW, chunks),
                                                 gs, (const float2*)ds, amax_c, (float*)workspace);
  RBU_CHECK_LAUNCH();
  rb_d_reduce_kernel<<<dim3(rbu_cdiv(2 * C, 128), N), 128, 0, st>>>((const float*)workspace, chunks, C, D);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// Between passes 2 and 3: ChannelAttention MLP backward (Main_Final.py:97-101), BatchNorm2 / shortcut-BN sums and the
// pass-3 coefficient arrays.  coef = float[(3*N + 1)*C] (c1, c0, cm per (n,c); cy per c); coef_s = float[3*C] (es, e0, ey).
extern "C" int rbu_rb_mid(const double* D, const float* g, const float* h_avg, const float* h_max, const float* u_avg,
                          const float* u_max, const float* nc_mean, const float* tv, const float* V1, const float* V2,
                          const float* scale2, const float* shift2, const float* mean2, const float* rstd2, int N, int HW,
                          int C, int Ch, float* scratch /* float[3*N*C + 2*N*Ch] */, float* dV1, float* dV2, float* sums2,
                          float* coef, const float* sums_s_raw, const float* scale_s, const float* mean_s,
                          const float* rstd_s, float* sums_s, float* coef_s, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(D && g && h_avg && h_max && u_avg && u_max && nc_mean && tv && V1 && V2 && scale2 && shift2 && mean2 && rstd2 &&
                    scratch && dV1 && dV2 && sums2 && coef && N > 0 && C > 0 && Ch > 0 && HW > 0 &&
                    (C + 2 * Ch) * 4 <= 48 * 1024, "rbu_rb_mid: bad arguments");
  RBU_CHECK_ARG(!sums_s_raw || (scale_s && mean_s && rstd_s && sums_s && coef_s), "rbu_rb_mid: projection-shortcut arguments missing");
  float* dt = scratch;
  float* du_avg = dt + (size_t)N * C;
  float* du_max = du_avg + (size_t)N * C;
  float* dh_avg = du_max + (size_t)N * C;
  float* dh_max = dh_avg + (size_t)N * Ch;
  ca_bwd_n_kernel<<<N, NT, (C + 2 * Ch) * sizeof(float), st>>>(D, scale2, shift2, g, h_avg, h_max, V1, V2, C, Ch, dt, dh_avg,
                                                               dh_max, du_avg, du_max);
  RBU_CHECK_LAUNCH();
  ca_bwd_w_kernel<<<rbu_cdiv((long)C * Ch, 32), 256, 0, st>>>(dt, dh_avg, dh_max, h_avg, h_max, u_avg, u_max, N, C, Ch,
                                                              dV1, dV2);
  RBU_CHECK_LAUNCH();
  float* c1 = coef;
  float* c0 = c1 + (size_t)N * C;
  float* cm = c0 + (size_t)N * C;
  float* cy = cm + (size_t)N * C;
  rb_coef_kernel<<<rbu_cdiv(C, 32), 256, 0, st>>>(D, g, du_avg, du_max, nc_mean, tv, scale2, mean2, rstd2, N, HW, C, sums2, c1,
                                                   c0, cm, cy, sums_s_raw, scale_s, mean_s, rstd_s, sums_s,
                                                   coef_s, coef_s ? coef_s + C : nullptr, coef_s ? coef_s + 2 * C : nullptr);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// pass 3: dy2 (and dys for a projection shortcut)
extern "C" int rbu_rb_bwd3(const void* de, int64_t de_ld, const void* y2, int64_t y2_ld, void* dy2, int64_t dy2_ld,
                           const void* ys, int64_t ys_ld, void* dys, int64_t dys_ld, int N, int HW, int C, const float* gs,
                           const float* ds, const int* amax_c, const int* nc_arg, const float* coef, const float* coef_s,
                           void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(de, de_ld) && VIEW_OK(y2, y2_ld) && VIEW_OK(dy2, dy2_ld) && CH_OK(C) && N > 0 && N <= 65535 && HW > 0 &&
                    gs && ds && amax_c && nc_arg && coef, "rbu_rb_bwd3: bad arguments");
  RBU_CHECK_ARG(!ys || (VIEW_OK(ys, ys_ld) && VIEW_OK(dys, dys_ld) && coef_s), "rbu_rb_bwd3: projection-shortcut arguments missing");
  int lg = 0;
  while ((1 << (lg + 1)) <= (C >> 3)) ++lg;
  const long items = (long)HW << lg;
  const long blocks = rbu_stream_blocks(items, NT * 2, N);
  const float* c1 = coef;
  const float* c0 = c1 + (size_t)N * C;
  const float* cm = c0 + (size_t)N * C;
  const float* cy = cm + (size_t)N * C;
  if (ys)
    rb_bwd3_kernel<true><<<dim3((unsigned)blocks, N), NT, 0, st>>>(
        (const bf16*)de, de_ld, (const bf16*)y2, y2_ld, (bf16*)dy2, dy2_ld, (const bf16*)ys, ys_ld, (bf16*)dys, dys_ld, HW, C, lg,
        gs, (const float2*)ds, amax_c, nc_arg, c1, c0, cm, cy, coef_s, coef_s + C, coef_s + 2 * C);
  else
    rb_bwd3_kernel<false><<<dim3((unsigned)blocks, N), NT, 0, st>>>(
        (const bf16*)de, de_ld, (const bf16*)y2, y2_ld, (bf16*)dy2, dy2_ld, nullptr, 0, nullptr, 0, HW, C, lg, gs,
        (const float2*)ds, amax_c, nc_arg, c1, c0, cm, cy, nullptr, nullptr, nullptr);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// BatchNorm(+ReLU)(+Dropout2d) backward: writes dx and sums[2C] = (dbeta, dgamma)
extern "C" int rbu_bn_bwd(const void* dy, int64_t dy_ld, const void* y, int64_t y_ld, void* dx, int64_t dx_ld, int N,
                          int HW, int C, const float* scale, const float* shift, const float* mean, const float* rstd,
                          const float* drop, int relu, float* sums, void* workspace, size_t workspace_bytes,
                          void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(dy, dy_ld) && VIEW_OK(y, y_ld) && VIEW_OK(dx, dx_ld) && CH_OK(C) && N > 0 && N <= 65535 && HW > 0 &&
                    scale && shift && mean && rstd && sums, "rbu_bn_bwd: bad arguments");
  const int chunks = bwd_chunks(N, HW, C);
  const int chunk_px = rbu_cdiv(HW, chunks);
  const size_t part_floats = (size_t)N * chunks * 2 * C;
  RBU_CHECK_ARG(workspace && workspace_bytes >= (part_floats + 2 * C + FOLD_FLOATS(2 * C)) * sizeof(float), "rbu_bn_bwd: workspace too small");
  float* part = (float*)workspace;
  float* coef = part + part_floats;
  const float invM = 1.f / ((float)N * (float)HW);
  bn_bwd_reduce_kernel<<<dim3(chunks, N), NT, 0, st>>>((const bf16*)dy, dy_ld, (const bf16*)y, y_ld, HW, C, chunk_px, scale,
                                                       shift, drop, relu, part);
  RBU_CHECK_LAUNCH();
  {
    const float* pp = part;
    int nb2 = N * chunks;
    long stride = 2 * C;
    int rc = colsum_fold(pp, nb2, stride, 2 * C, coef + 2 * C, st);
    if (rc) return rc;
    bn_bwd_final_kernel<<<rbu_cdiv(C, 32), 256, 0, st>>>(pp, nb2, C, scale, mean, rstd, invM, sums, coef);
    RBU_CHECK_LAUNCH();
  }
  int lg = 0;
  while ((1 << (lg + 1)) <= (C >> 3)) ++lg;
  const long items = (long)HW << lg;
  const long blocks = rbu_stream_blocks(items, NT * 4, N);
  bn_bwd_apply_kernel<<<dim3((unsigned)blocks, N), NT, 0, st>>>((const bf16*)dy, dy_ld, (const bf16*)y, y_ld, (bf16*)dx, dx_ld,
                                                                HW, C, lg, scale, shift, drop, relu, coef);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

// AttentionGate backward.  Outputs: dskip view (= da*psi), dyg/dyx views, sums_f[4][F] (dwpsi, dbeta_g(=dbeta_x),
// dgamma_g, dgamma_x), sums_psi[2] (dbeta_psi, dgamma_psi).
extern "C" int rbu_ag_bwd(const void* da, int64_t da_ld, const void* skip, int64_t s_ld, void* dskip, int64_t ds_ld,
                          const void* yg, int64_t yg_ld, const void* yx, int64_t yx_ld, void* dyg, int64_t dyg_ld,
                          void* dyx, int64_t dyx_ld, int N, int HW, int C, int F, const float* psi, const float* q0,
                          const float* stats, const float* Ag, const float* Bg, const float* Ax, const float* Bx,
                          const float* mg, const float* rg, const float* mx, const float* rx, const float* wpsi,
                          float* dq, float* sums_psi, float* sums_f, void* workspace, size_t workspace_bytes,
                          void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(da, da_ld) && VIEW_OK(skip, s_ld) && VIEW_OK(dskip, ds_ld) && VIEW_OK(yg, yg_ld) && VIEW_OK(yx, yx_ld) &&
                    VIEW_OK(dyg, dyg_ld) && VIEW_OK(dyx, dyx_ld) && CH_OK(C) && CH_OK(F) && N > 0 && N <= 65535 && HW > 0,
                "rbu_ag_bwd: bad views");
  RBU_CHECK_ARG(psi && q0 && stats && Ag && Bg && Ax && Bx && mg && rg && mx && rx && wpsi && dq && sums_psi && sums_f,
                "rbu_ag_bwd: null pointer");
  const float invM = 1.f / ((float)N * (float)HW);
  float* part = (float*)workspace;
  {
    const int chunks = bwd_chunks(N, HW, C);
    RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)N * chunks * 2 * sizeof(float), "rbu_ag_bwd: workspace too small");
    ag_bwd1_kernel<<<dim3(chunks, N), NT, 0, st>>>((const bf16*)da, da_ld, (const bf16*)skip, s_ld, (bf16*)dskip, ds_ld, HW,
                                                   C, rbu_cdiv(HW, chunks), psi, q0, stats, dq, part);
    RBU_CHECK_LAUNCH();
    const float* pp = part;
    int nb2 = N * chunks;
    long stride = 2;
    RBU_CHECK_ARG(workspace_bytes >= ((size_t)N * chunks * 2 + FOLD_FLOATS(2)) * sizeof(float), "rbu_ag_bwd: workspace too small");
    int rc = colsum_fold(pp, nb2, stride, 2, part + (size_t)N * chunks * 2, st);
    if (rc) return rc;
    colsum_kernel<<<1, 256, 0, st>>>(pp, nb2, 2, stride, sums_psi, 1.f);
    RBU_CHECK_LAUNCH();
  }
  {
    const int chunks = bwd_chunks(N, HW, F);
    const int chunk_px = rbu_cdiv(HW, chunks);
    const size_t part_floats = (size_t)N * chunks * 4 * F;
    RBU_CHECK_ARG(workspace_bytes >= (part_floats + 4 * F + FOLD_FLOATS(4 * F)) * sizeof(float), "rbu_ag_bwd: workspace too small");
    float* coef = part + part_floats;
    ag_bwd2_kernel<<<dim3(chunks, N), NT, 0, st>>>((const bf16*)yg, yg_ld, (const bf16*)yx, yx_ld, HW, F, chunk_px, Ag, Bg, Ax,
                                                   Bx, wpsi, dq, q0, stats, sums_psi, invM, part);
    RBU_CHECK_LAUNCH();
    {
      const float* pp = part;
      int nb2 = N * chunks;
      long stride = 4 * F;
      int rc = colsum_fold(pp, nb2, stride, 4 * F, coef + 4 * F, st);
      if (rc) return rc;
      ag_bwd_final_kernel<<<rbu_cdiv(F, 32), 256, 0, st>>>(pp, nb2, F, Ag, Ax, mg, rg, mx, rx, invM, sums_f, coef);
      RBU_CHECK_LAUNCH();
    }
    int lg = 0;
    while ((1 << (lg + 1)) <= (F >> 3)) ++lg;
    const long items = (long)HW << lg;
    const long blocks = rbu_stream_blocks(items, NT * 2, N);
    ag_bwd3_kernel<<<dim3((unsigned)blocks, N), NT, 0, st>>>((const bf16*)yg, yg_ld, (const bf16*)yx, yx_ld, (bf16*)dyg, dyg_ld,
                                                             (bf16*)dyx, dyx_ld, HW, F, lg, Ag, Bg, Ax, Bx, wpsi, dq, q0, stats,
                                                             sums_psi, invM, coef);
    RBU_CHECK_LAUNCH();
  }
  return RBU_OK;
}

extern "C" int rbu_maxpool2x2_bwd(const void* x, int64_t x_ld, const void* dy, int64_t dy_ld, void* dx, int64_t dx_ld,
                                  int N, int Ho, int Wo, int C, int accumulate, void* stream_) {
  RBU_CHECK_ARG(VIEW_OK(x, x_ld) && VIEW_OK(dy, dy_ld) && VIEW_OK(dx, dx_ld) && N > 0 && Ho > 0 && Wo > 0 && C % 8 == 0,
                "rbu_maxpool2x2_bwd: bad arguments");
  maxpool_bwd_kernel<<<grid1d((long)N * Ho * Wo * (C >> 3), NT), NT, 0, (cudaStream_t)stream_>>>(
      (const bf16*)x, x_ld, (const bf16*)dy, dy_ld, (bf16*)dx, dx_ld, N, Ho, Wo, C, accumulate);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_chan_sum(const void* x, int64_t ld, int64_t P, int C, float* out, void* workspace,
                            size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(VIEW_OK(x, ld) && out && CH_OK(C) && P > 0, "rbu_chan_sum: bad arguments");
  int ppb;
  const int blocks = flat_blocks(P, C, &ppb);
  RBU_CHECK_ARG(workspace && workspace_bytes >= (size_t)blocks * C * sizeof(float), "rbu_chan_sum: workspace too small");
  chan_sum_kernel<<<blocks, NT, 0, st>>>((const bf16*)x, ld, P, C, ppb, (float*)workspace);
  RBU_CHECK_LAUNCH();
  const float* pp = (const float*)workspace;
  int nb2 = blocks;
  long stride = C;
  RBU_CHECK_ARG(workspace_bytes >= ((size_t)blocks * C + FOLD_FLOATS(C)) * sizeof(float), "rbu_chan_sum: workspace too small");
  int rc = colsum_fold(pp, nb2, stride, C, (float*)workspace + (size_t)blocks * C, st);
  if (rc) return rc;
  colsum_kernel<<<rbu_cdiv(C, 32), 256, 0, st>>>(pp, nb2, C, stride, out, 1.f);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
