// Resizing of uint8 images and masks, bit-exact with the third-party calls of the reference:
//   mode 0  Pillow Image.resize(BILINEAR) = torchvision transforms.Resize on PIL images (Main_Final.py:697-701,
//           predict_coastline.py:386-392): Pillow's Resample.c, 8 bits per sample -- triangle filter widened by the
//           downscale factor (antialiasing), weights normalised in double and rounded to 22 fraction bits, horizontal
//           pass first with a uint8 intermediate, then the vertical pass;
//   mode 1  Pillow Image.resize(NEAREST) (mask resize, Main_Final.py:44-54): Geometry.c's affine scaler, whose source
//           coordinate is ACCUMULATED (xo = a/2; xo += a), which differs from (int)(a*(o+0.5)) for e.g. 4 -> 333;
//   mode 2  cv2.resize(INTER_NEAREST) (predicted mask back to scene size, predict_coastline.py:583-602):
//           idx = min(floor(o * (1.0 / ((double)out / in))), in - 1).
// One launch per call for a batch of sources of different sizes (device descriptor array, grid = tiles x images).
// The double expressions use explicitly rounded intrinsics so nvcc cannot contract them into FMAs: the tap window and
// the weights depend on every rounding.
#include "rbu_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kPrec = 22;                  // Resample.c PRECISION_BITS (32 - 8 - 2)
// Bilinear output tile: 64 columns x 32 rows, one column and 8 rows (interleaved by 4) per thread.  At a 2x downscale a
// tile reads 68 x 132 source pixels for 32 x 64 outputs: 10 % of the source is read twice.
constexpr int kTW = 64;
constexpr int kTH = 32;
constexpr int kRowsPerThread = kTH / (kThreads / kTW);
constexpr int kMaxChunkRows = 128;         // source rows of the uint8 intermediate held in shared memory at once
constexpr int kNearestRows = 16;           // output rows per CTA of the nearest-neighbour gathers
constexpr size_t kMaxSmem = 200 * 1024;    // dynamic shared memory of one CTA (the bilinear plan at 255 taps is 123 KB)

// Pillow's ksize for one axis: 2 * ceil(support) + 1 with support = max(in / out, 1).
__host__ __device__ inline int bilinear_ksize(int n_in, int n_out) {
#ifdef __CUDA_ARCH__
  double scale = __ddiv_rn((double)n_in, (double)n_out);
#else
  double scale = (double)n_in / (double)n_out;
#endif
  if (scale < 1.0) scale = 1.0;
  return 2 * (int)ceil(scale) + 1;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc (triangle filter, support 1) for output index o: writes the
// int32 weights to k[0..n) and returns the first tap; *n_out is the tap count (xmax - xmin).
__device__ int bilinear_taps(int n_in, int n_out, int o, int* k, int* n_taps) {
  const double scale = __ddiv_rn((double)n_in, (double)n_out);
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = fs;                                    // 1.0 * filterscale
  const double ss = __ddiv_rn(1.0, fs);
  const double center = __dmul_rn(__dadd_rn((double)o, 0.5), scale);
  int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, support), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, support), 0.5));
  if (xmax > n_in) xmax = n_in;
  const int n = xmax - xmin;
  double ww = 0.0;
  for (int x = 0; x < n; ++x) {
    const double t = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
    ww = __dadd_rn(ww, t < 1.0 ? __dsub_rn(1.0, t) : 0.0);
  }
  for (int x = 0; x < n; ++x) {
    const double t = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
    double w = t < 1.0 ? __dsub_rn(1.0, t) : 0.0;
    if (ww != 0.0) w = __ddiv_rn(w, ww);
    k[x] = __double2int_rz(__dadd_rn(0.5, __dmul_rn(w, (double)(1 << kPrec))));     // w >= 0 for this filter
  }
  *n_taps = n;
  return xmin;
}

__device__ __forceinline__ int clip8(int acc) { return min(acc >> kPrec, 255); }      // acc >= 0: weights are >= 0

// Two-pass bilinear resize of one 32 x 64 output tile of image blockIdx.y.  The prologue computes the tile's column and
// row weights into shared memory; the source rows the tile needs are then processed in chunks of at most `chunk` rows:
// horizontal pass from global memory into a uint8 chunk in shared memory, vertical pass from there into int32
// registers.  Integer sums are associative, so chunking changes nothing in the result.
template <int C>
__global__ void __launch_bounds__(kThreads)
resize_bilinear_kernel(const rbu_resize_src* __restrict__ srcs, int oh, int ow, int kh_stride, int kv_stride, int chunk,
                       uint8_t* __restrict__ out) {
  extern __shared__ int smem[];
  int* kh = smem;                                   // [kTW][kh_stride]
  int* kv = kh + kTW * kh_stride;                   // [kTH][kv_stride]
  int* xlo = kv + kTH * kv_stride;
  int* xn = xlo + kTW;
  int* ylo = xn + kTW;
  int* yn = ylo + kTH;
  uint8_t* tmp = reinterpret_cast<uint8_t*>(yn + kTH);      // [chunk][kTW * C]

  const rbu_resize_src d = srcs[blockIdx.y];
  // a descriptor beyond the sizes the launch was planned for (or empty) is skipped, never read out of bounds
  if (d.src == nullptr || d.H <= 0 || d.W <= 0 || bilinear_ksize(d.W, ow) > kh_stride ||
      bilinear_ksize(d.H, oh) > kv_stride)
    return;
  const int ntx = (ow + kTW - 1) / kTW;
  const int ox0 = (blockIdx.x % ntx) * kTW;
  const int oy0 = (blockIdx.x / ntx) * kTH;
  const int ncols = min(kTW, ow - ox0);
  const int nrows = min(kTH, oh - oy0);
  const int tid = threadIdx.x;
  if (tid < ncols) {
    xlo[tid] = bilinear_taps(d.W, ow, ox0 + tid, kh + tid * kh_stride, &xn[tid]);
  } else if (tid >= kTW && tid - kTW < nrows) {
    const int r = tid - kTW;
    ylo[r] = bilinear_taps(d.H, oh, oy0 + r, kv + r * kv_stride, &yn[r]);
  }
  __syncthreads();
  const int y_begin = ylo[0];
  const int y_end = ylo[nrows - 1] + yn[nrows - 1];       // tap windows are monotone in the output index

  const int o = tid % kTW;
  const int rg = tid / kTW;
  int acc[kRowsPerThread][C];
#pragma unroll
  for (int i = 0; i < kRowsPerThread; ++i)
#pragma unroll
    for (int c = 0; c < C; ++c) acc[i][c] = 1 << (kPrec - 1);

  for (int c0 = y_begin; c0 < y_end; c0 += chunk) {
    const int c1 = min(c0 + chunk, y_end);
    const int n_elems = (c1 - c0) * kTW * C;
    for (int idx = tid; idx < n_elems; idx += kThreads) {
      const int r = idx / (kTW * C);
      const int e = idx - r * (kTW * C);
      const int oc = e / C;
      if (oc < ncols) {
        const int ch = e - oc * C;
        const uint8_t* s = d.src + (long long)(c0 + r) * d.row_pitch + xlo[oc] * C + ch;
        const int* k = kh + oc * kh_stride;
        int a = 1 << (kPrec - 1);
        for (int j = 0; j < xn[oc]; ++j) a += (int)__ldg(s + j * C) * k[j];
        tmp[idx] = (uint8_t)clip8(a);
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kRowsPerThread; ++i) {
      const int lr = rg + i * (kThreads / kTW);
      if (lr < nrows) {
        const int lo = ylo[lr];
        const int j0 = max(c0 - lo, 0);
        const int j1 = min(c1 - lo, yn[lr]);
        const int* k = kv + lr * kv_stride;
        for (int j = j0; j < j1; ++j) {
          const uint8_t* t = tmp + (lo + j - c0) * (kTW * C) + o * C;
#pragma unroll
          for (int c = 0; c < C; ++c) acc[i][c] += (int)t[c] * k[j];
        }
      }
    }
    __syncthreads();
  }

  if (o >= ncols) return;
  const int ox = ox0 + o;
#pragma unroll
  for (int i = 0; i < kRowsPerThread; ++i) {
    const int lr = rg + i * (kThreads / kTW);
    if (lr >= nrows) continue;
    uint8_t* p = out + (((long long)blockIdx.y * oh + oy0 + lr) * ow + ox) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) p[c] = (uint8_t)clip8(acc[i][c]);
  }
}

// Nearest-neighbour gather of kNearestRows full output rows of image blockIdx.y.  The index tables live in shared
// memory.  PILLOW: Pillow's coordinate is a loop-carried double sum, so one thread per axis walks it in the prologue
// (ow + oy0 + kNearestRows dependent adds per CTA -- cheap at the 512-pixel mask sizes the reference resizes to); an
// index that reaches the source size is an output pixel Pillow leaves at 0 (-1 here).  Otherwise OpenCV's closed form,
// one index per thread.
template <int C, bool PILLOW>
__global__ void __launch_bounds__(kThreads)
resize_nearest_kernel(const rbu_resize_src* __restrict__ srcs, int oh, int ow, uint8_t* __restrict__ out) {
  extern __shared__ int smem[];
  int* xidx = smem;                    // [ow]
  int* yidx = smem + ow;               // [kNearestRows]
  const rbu_resize_src d = srcs[blockIdx.y];
  if (d.src == nullptr || d.H <= 0 || d.W <= 0) return;
  const int oy0 = blockIdx.x * kNearestRows;
  const int nrows = min(kNearestRows, oh - oy0);
  const int tid = threadIdx.x;
  if (PILLOW) {
    if (tid == 0) {
      const double a = __ddiv_rn((double)d.W, (double)ow);
      double xo = __dmul_rn(a, 0.5);
      for (int x = 0; x < ow; ++x) {
        const int i = __double2int_rz(xo);
        xidx[x] = i < d.W ? i : -1;
        xo = __dadd_rn(xo, a);
      }
    } else if (tid == 32) {
      const double a = __ddiv_rn((double)d.H, (double)oh);
      double yo = __dmul_rn(a, 0.5);
      for (int y = 0; y < oy0 + nrows; ++y) {
        if (y >= oy0) {
          const int i = __double2int_rz(yo);
          yidx[y - oy0] = i < d.H ? i : -1;
        }
        yo = __dadd_rn(yo, a);
      }
    }
  } else {
    const double fx = __ddiv_rn(1.0, __ddiv_rn((double)ow, (double)d.W));
    const double fy = __ddiv_rn(1.0, __ddiv_rn((double)oh, (double)d.H));
    for (int x = tid; x < ow; x += kThreads) xidx[x] = min((int)floor(__dmul_rn((double)x, fx)), d.W - 1);
    if (tid < nrows) yidx[tid] = min((int)floor(__dmul_rn((double)(oy0 + tid), fy)), d.H - 1);
  }
  __syncthreads();
  const int row_elems = ow * C;
  for (int r = 0; r < nrows; ++r) {
    const int y = yidx[r];
    const uint8_t* srow = d.src + (long long)(y < 0 ? 0 : y) * d.row_pitch;
    uint8_t* orow = out + ((long long)blockIdx.y * oh + oy0 + r) * row_elems;
    for (int e = tid; e < row_elems; e += kThreads) {
      const int x = xidx[e / C];
      orow[e] = (y < 0 || x < 0) ? 0 : __ldg(srow + x * C + e % C);
    }
  }
}

struct BilinearPlan {
  int kh, kv, chunk;
  size_t smem;
};

BilinearPlan plan_bilinear(int C, int max_h, int max_w, int oh, int ow) {
  BilinearPlan p;
  p.kh = bilinear_ksize(max_w, ow);
  p.kv = bilinear_ksize(max_h, oh);
  // source rows one tile needs: 32 output rows' windows at the largest vertical scale, plus both filter tails
  const double sv = (double)max_h / oh;
  const long span = (long)ceil(kTH * (sv > 1.0 ? sv : 1.0)) + p.kv + 1;
  p.chunk = (int)(span < kMaxChunkRows ? span : kMaxChunkRows);
  p.smem = (size_t)(kTW * p.kh + kTH * p.kv + 2 * kTW + 2 * kTH) * sizeof(int) + (size_t)p.chunk * kTW * C;
  return p;
}

template <int C>
int launch_bilinear(const rbu_resize_src* srcs, int B, int max_h, int max_w, int oh, int ow, uint8_t* out,
                    cudaStream_t stream) {
  const BilinearPlan p = plan_bilinear(C, max_h, max_w, oh, ow);
  static std::atomic<unsigned long long> done{0};
  if (rbu_first_use_on_device(&done))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(resize_bilinear_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kMaxSmem));
  const long tiles = (long)((ow + kTW - 1) / kTW) * ((oh + kTH - 1) / kTH);
  resize_bilinear_kernel<C><<<dim3((unsigned)tiles, B), kThreads, p.smem, stream>>>(srcs, oh, ow, p.kh, p.kv,
                                                                                           p.chunk, out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

template <int C>
int launch_nearest(const rbu_resize_src* srcs, int B, int oh, int ow, int mode, uint8_t* out, cudaStream_t stream) {
  const size_t smem = (size_t)(ow + kNearestRows) * sizeof(int);
  const dim3 grid((unsigned)((oh + kNearestRows - 1) / kNearestRows), B);
  if (mode == 1) {
    static std::atomic<unsigned long long> done{0};
    if (rbu_first_use_on_device(&done))
      RBU_CHECK_CUDA(cudaFuncSetAttribute(resize_nearest_kernel<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          kMaxSmem));
    resize_nearest_kernel<C, true><<<grid, kThreads, smem, stream>>>(srcs, oh, ow, out);
  } else {
    static std::atomic<unsigned long long> done{0};
    if (rbu_first_use_on_device(&done))
      RBU_CHECK_CUDA(cudaFuncSetAttribute(resize_nearest_kernel<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          kMaxSmem));
    resize_nearest_kernel<C, false><<<grid, kThreads, smem, stream>>>(srcs, oh, ow, out);
  }
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

int check_common(const char* fn, const rbu_resize_src* srcs, int B, int max_h, int max_w, int oh, int ow) {
  RBU_CHECK_ARG(srcs && B > 0 && B <= 65535 && max_h > 0 && max_w > 0 && oh > 0 && ow > 0, "%s: bad arguments", fn);
  return RBU_OK;
}

int check_bilinear(const char* fn, int max_h, int max_w, int oh, int ow) {
  const int taps = bilinear_ksize(max_w, ow) > bilinear_ksize(max_h, oh) ? bilinear_ksize(max_w, ow)
                                                                          : bilinear_ksize(max_h, oh);
  if (taps > RBU_RESIZE_MAX_TAPS) {
    rbu_set_error("%s: a %dx%d -> %dx%d bilinear resize needs %d taps per output (at most %d: downscales up to %dx)",
                  fn, max_h, max_w, oh, ow, taps, RBU_RESIZE_MAX_TAPS, (RBU_RESIZE_MAX_TAPS - 1) / 2);
    return RBU_ERR_UNSUPPORTED;
  }
  return RBU_OK;
}

}  // namespace

extern "C" int rbu_resize_u8(const rbu_resize_src* srcs_device, int B, int C, int max_h, int max_w, int oh, int ow,
                             int mode, uint8_t* out, void* stream) {
  if (int rc = check_common("rbu_resize_u8", srcs_device, B, max_h, max_w, oh, ow)) return rc;
  RBU_CHECK_ARG(out && (C == 1 || C == 3), "rbu_resize_u8: C must be 1 or 3");
  RBU_CHECK_ARG(mode >= 0 && mode <= 2, "rbu_resize_u8: mode must be 0 (bilinear), 1 (Pillow nearest) or 2 (cv2 nearest)");
  cudaStream_t s = (cudaStream_t)stream;
  if (mode == 0) {
    if (int rc = check_bilinear("rbu_resize_u8", max_h, max_w, oh, ow)) return rc;
    return C == 1 ? launch_bilinear<1>(srcs_device, B, max_h, max_w, oh, ow, out, s)
                  : launch_bilinear<3>(srcs_device, B, max_h, max_w, oh, ow, out, s);
  }
  if ((size_t)(ow + kNearestRows) * sizeof(int) > kMaxSmem) {
    rbu_set_error("rbu_resize_u8: output width %d exceeds the nearest-neighbour index table", ow);
    return RBU_ERR_UNSUPPORTED;
  }
  return C == 1 ? launch_nearest<1>(srcs_device, B, oh, ow, mode, out, s)
                : launch_nearest<3>(srcs_device, B, oh, ow, mode, out, s);
}
