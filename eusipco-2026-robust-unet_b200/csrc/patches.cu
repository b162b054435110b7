// Patch sampling for native-resolution training: crop ph x pw patches out of whole scenes resident in HBM, apply one of
// the eight flips / 90-degree rotations (the dihedral group), and write the network input (preprocess_pixel, bit-exact
// with rbu_preprocess) and the mask patch.  A job's origin is either host-drawn or centred on the k-th nonzero pixel of
// the scene's focus mask (nnU-Net's foreground oversampling, MONAI's RandCropByPosNegLabel).
//
// One CTA owns one kTile x kTile output tile of one patch:
//   1. warp 0 resolves the patch origin (for a focus job: a 32-ary warp search over focus_rows for the row, then a warp
//      scan of that row's nonzero counts for the column) -- every CTA of a patch repeats it, which keeps a call to one
//      launch;
//   2. the CTA stages the source rectangle its tile reads (a transposing op reads it column-wise) in shared memory, one
//      warp per source row, so the uint8 HWC rows are read coalesced;
//   3. one thread per output pixel reads the transformed pixel from shared memory and writes the nc fp32 planes and the
//      mask byte, a warp covering 32 consecutive output columns (coalesced stores).
// Offsets into scenes and outputs are 64-bit: a scene may exceed 2 GiB.
#include "preprocess.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kTile = 64;
constexpr int kImgStride = 3 * kTile + 4;   // bytes per staged image row: 49 words (odd), so column reads are
constexpr int kMskStride = kTile + 4;       // conflict-free; mask rows 17 words
static_assert(sizeof(rbu_patch_src) == 64 && sizeof(rbu_patch_job) == 32, "patches.py builds these tables with numpy");

// focus_rows[H] > 0 and 0 <= k < focus_rows[H]: the (row, column) of the k-th nonzero focus pixel in row-major order.
// Called by one whole warp; every lane returns the same pair.  An inconsistent focus_rows table cannot make it read
// outside the scene: the column then falls back to 0.
__device__ void kth_focus_pixel(const uint8_t* __restrict__ focus, long long pitch, const long long* __restrict__ rows,
                                int H, int W, long long k, int& py, int& px) {
  const int lane = threadIdx.x & 31;
  // rows[lo] <= k < rows[hi]; each step probes 32 points of (lo, hi) at once.  rows is non-decreasing, so the probes
  // with rows[p] <= k form a prefix of the lanes.
  int lo = 0, hi = H;
  while (hi - lo > 1) {
    const int p = lo + (int)((long long)(hi - lo) * (lane + 1) / 33);
    const bool le = __ldg(rows + p) <= k;
    const unsigned m = __ballot_sync(0xffffffffu, le);
    const int nlo = m ? __shfl_sync(0xffffffffu, p, 31 - __clz(m)) : lo;
    const int nhi = ~m ? __shfl_sync(0xffffffffu, p, __ffs(~m) - 1) : hi;
    lo = max(lo, nlo);
    hi = min(hi, nhi);
  }
  py = lo;
  const int kk = (int)(k - __ldg(rows + lo));         // < W
  // lane l counts the nonzeros of columns [l*C, (l+1)*C); an inclusive warp scan finds the lane holding the kk-th
  const uint8_t* row = focus + (long long)lo * pitch;
  const int C = (W + 31) / 32;
  const int c0 = min(W, lane * C), c1 = min(W, c0 + C);
  int cnt = 0;
  for (int c = c0; c < c1; ++c) cnt += __ldg(row + c) != 0;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const int excl = incl - cnt;
  const bool mine = excl <= kk && kk < incl;
  int col = 0;
  if (mine) {
    int need = kk - excl;
    for (int c = c0; c < c1; ++c)
      if (__ldg(row + c) != 0 && need-- == 0) {
        col = c;
        break;
      }
  }
  const unsigned m = __ballot_sync(0xffffffffu, mine);
  px = m ? __shfl_sync(0xffffffffu, col, __ffs(m) - 1) : 0;
}

__global__ void __launch_bounds__(kThreads)
sample_patches_kernel(const rbu_patch_src* __restrict__ srcs, int S, const rbu_patch_job* __restrict__ jobs, int ph,
                      int pw, int tiles_x, int tiles_per_patch, int nc, float* __restrict__ images_out,
                      uint8_t* __restrict__ masks_out, int* __restrict__ jobs_out) {
  __shared__ uint8_t s_img[kTile * kImgStride];
  __shared__ uint8_t s_msk[kTile * kMskStride];
  __shared__ int s_org[3];                           // valid, y, x
  const int b = blockIdx.x / tiles_per_patch;
  const int tile = blockIdx.x - b * tiles_per_patch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const rbu_patch_job job = jobs[b];
  const int op = job.op;
  const bool tr = op & 4, fh = op & 2, fw = op & 1;
  const int wh = tr ? pw : ph, ww = tr ? ph : pw;    // the window read from the scene

  if (warp == 0) {
    bool valid = job.scene >= 0 && job.scene < S && op >= 0 && op < 8;
    int y = job.y0, x = job.x0;
    if (valid) {
      const rbu_patch_src& s = srcs[job.scene];
      valid = wh <= s.H && ww <= s.W;
      const long long total = job.focus && s.focus && s.focus_rows ? __ldg(s.focus_rows + s.H) : 0;
      if (valid && total > 0) {
        int py, px;
        kth_focus_pixel(s.focus, s.focus_pitch, s.focus_rows, s.H, s.W, (long long)((unsigned long long)job.r % total),
                        py, px);
        y = min(max(py - wh / 2, 0), s.H - wh);
        x = min(max(px - ww / 2, 0), s.W - ww);
      }
      valid = valid && y >= 0 && y <= s.H - wh && x >= 0 && x <= s.W - ww;
    }
    if (lane == 0) {
      s_org[0] = valid;
      s_org[1] = y;
      s_org[2] = x;
      if (jobs_out && tile == 0) {
        int* o = jobs_out + 4LL * b;
        o[0] = valid ? job.scene : -1;
        o[1] = valid ? y : -1;
        o[2] = valid ? x : -1;
        o[3] = valid ? op : -1;
      }
    }
  }
  __syncthreads();
  if (!s_org[0]) return;                             // a job the scene cannot hold: its patch is left unwritten
  const rbu_patch_src& s = srcs[job.scene];
  const int y = s_org[1], x = s_org[2];

  // output tile rows [ti, ti + ni), columns [tj, tj + nj); after the flips they read window rows / columns starting at
  // il / jl, and the transpose swaps the two
  const int ty = tile / tiles_x;
  const int ti = ty * kTile, tj = (tile - ty * tiles_x) * kTile;
  const int ni = min(kTile, ph - ti), nj = min(kTile, pw - tj);
  const int il = fh ? ph - ti - ni : ti, jl = fw ? pw - tj - nj : tj;
  const int r0 = tr ? jl : il, c0 = tr ? il : jl;    // the source rectangle, relative to the window origin
  const int rh = tr ? nj : ni, rw = tr ? ni : nj;

  for (int r = warp; r < rh; r += kThreads / 32) {
    const long long sy = (long long)y + r0 + r;
    const uint8_t* irow = s.image + sy * s.image_pitch + 3LL * (x + c0);
    const uint8_t* mrow = s.mask + sy * s.mask_pitch + (x + c0);
    uint8_t v[3 * kTile / 32 + kTile / 32];
#pragma unroll
    for (int q = 0; q < 3 * kTile / 32; ++q) {
      const int c = lane + 32 * q;
      v[q] = c < 3 * rw ? __ldcs(irow + c) : 0;
    }
#pragma unroll
    for (int q = 0; q < kTile / 32; ++q) {
      const int c = lane + 32 * q;
      v[3 * kTile / 32 + q] = c < rw ? __ldcs(mrow + c) : 0;
    }
#pragma unroll
    for (int q = 0; q < 3 * kTile / 32; ++q) s_img[r * kImgStride + lane + 32 * q] = v[q];
#pragma unroll
    for (int q = 0; q < kTile / 32; ++q) s_msk[r * kMskStride + lane + 32 * q] = v[3 * kTile / 32 + q];
  }
  __syncthreads();

  const long long plane = (long long)ph * pw;
  float* img_b = images_out + (long long)b * nc * plane;
  uint8_t* msk_b = masks_out + (long long)b * plane;
  for (int p = threadIdx.x; p < kTile * kTile; p += kThreads) {
    const int di = p / kTile, dj = p - di * kTile;
    if (di >= ni || dj >= nj) continue;
    const int i = ti + di, j = tj + dj;
    const int iw = (fh ? ph - 1 - i : i) - il, jw = (fw ? pw - 1 - j : j) - jl;
    const int a = tr ? jw : iw, c = tr ? iw : jw;  // row / column inside the staged rectangle
    const uint8_t* px = s_img + a * kImgStride + 3 * c;
    const uint8_t rgb[3] = {px[0], px[1], px[2]};
    const long long o = (long long)i * pw + j;
    preprocess_pixel(rgb, nc, img_b + o, plane);
    msk_b[o] = s_msk[a * kMskStride + c];
  }
}

}  // namespace

extern "C" int rbu_sample_patches(const rbu_patch_src* srcs_device, int S, const rbu_patch_job* jobs_device, int B,
                                  int ph, int pw, int n_channels, float* images_out, uint8_t* masks_out, int* jobs_out,
                                  void* stream) {
  RBU_CHECK_ARG(srcs_device && jobs_device && images_out && masks_out, "rbu_sample_patches: null pointer");
  RBU_CHECK_ARG(S > 0 && B > 0 && ph > 0 && pw > 0, "rbu_sample_patches: bad sizes (S %d, B %d, patch %dx%d)", S, B, ph,
                pw);
  RBU_CHECK_ARG(n_channels == 3 || n_channels == 4 || n_channels == 6,
                "rbu_sample_patches: n_channels must be 3, 4 or 6, got %d", n_channels);
  const int tiles_x = (pw + kTile - 1) / kTile;
  const long long tiles = (long long)((ph + kTile - 1) / kTile) * tiles_x;
  RBU_CHECK_ARG(tiles * B < (1LL << 31), "rbu_sample_patches: %lld tiles per call (at most 2^31 - 1)", tiles * B);
  sample_patches_kernel<<<(unsigned)(tiles * B), kThreads, 0, (cudaStream_t)stream>>>(
      srcs_device, S, jobs_device, ph, pw, tiles_x, (int)tiles, n_channels, images_out, masks_out, jobs_out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
