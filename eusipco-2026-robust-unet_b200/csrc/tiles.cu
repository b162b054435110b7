// Sliding-window (tiled) inference of a whole scene: cut overlapping tiles out of an fp32 NCHW scene, and blend the
// network's per-tile outputs back with a separable Gaussian window (nnU-Net / MONAI sliding-window inference).
//   tile_gather_kernel  scene -> [Tb][nc][th][tw] for tiles t0 .. t0+Tb-1; one warp per tile row, so the reads of a
//                       scene row and the writes of a tile row are coalesced.  Rows / columns beyond the scene (a tile
//                       larger than the scene, by < 16 on the Python side) are reflected: F.pad(mode="reflect").
//   tile_blend_kernel   for each output pixel, a GATHER over the tiles that cover it (no atomics, bit-deterministic):
//                       w = wy[y - oy_i] * wx[x - ox_j];  num_k += w * v_k;  den += w;  out_k = num_k / den
//                       over i ascending (outer), j ascending (inner), every step a separately rounded fp32 op, so an
//                       fp32 CPU restatement in the same order (oracle/tiled_ref.py) matches bit for bit.  The K sums
//                       stay in registers, so the labels (threshold at K = 1, arg-max at K >= 2) need no second pass.
// Each tile element is read exactly once by the blend, so the tile values are streaming loads.
#include "rbu_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxK = 32;

int grid_for(long items, int per_block) {
  long b = (items + per_block - 1) / per_block;
  const long cap = (long)rbu_num_sms() * 8;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// F.pad(mode="reflect") index for one bounce; the clamp only keeps an inconsistent origin table inside the scene
__device__ __forceinline__ int reflect_index(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return min(max(i, 0), n - 1);
}

__global__ void __launch_bounds__(kThreads)
tile_gather_kernel(const float* __restrict__ x, int nc, int H, int W, const int* __restrict__ oy,
                   const int* __restrict__ ox, int nx, int th, int tw, int t0, int rows, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (kThreads / 32);
  for (int row = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); row < rows; row += warps) {
    const int r = row % th;
    const int bc = row / th;
    const int c = bc % nc;
    const int t = t0 + bc / nc;
    const int iy = t / nx;
    const int ix = t - iy * nx;
    const int yy = reflect_index(__ldg(oy + iy) + r, H);
    const int x0 = __ldg(ox + ix);
    const float* src = x + ((long long)c * H + yy) * W;
    float* dst = out + (long long)row * tw;
    for (int col = lane; col < tw; col += 32) dst[col] = __ldg(src + reflect_index(x0 + col, W));
  }
}

template <int KB>
__global__ void __launch_bounds__(kThreads)
tile_blend_kernel(const float* __restrict__ tiles, int K, int H, int W, const int* __restrict__ oy,
                  const int* __restrict__ ox, int ny, int nx, int th, int tw, const int* __restrict__ row_first,
                  const int* __restrict__ row_count, const int* __restrict__ col_first,
                  const int* __restrict__ col_count, const float* __restrict__ wy, const float* __restrict__ wx,
                  float threshold, float* __restrict__ out, uint8_t* __restrict__ labels) {
  const int segs = (W + kThreads - 1) / kThreads;
  const long long plane = (long long)th * tw;
  const long long HW = (long long)H * W;
  for (int s = blockIdx.x; s < H * segs; s += gridDim.x) {       // H * segs < 2^31: checked by the entry point
    const int y = s / segs;
    const int x = (s - y * segs) * kThreads + threadIdx.x;
    if (x >= W) continue;
    const int i0 = __ldg(row_first + y), ni = __ldg(row_count + y);
    const int j0 = __ldg(col_first + x), nj = __ldg(col_count + x);
    float num[KB];
#pragma unroll
    for (int k = 0; k < KB; ++k) num[k] = 0.f;
    float den = 0.f;
    for (int a = 0; a < ni; ++a) {
      const int i = i0 + a;
      if (i < 0 || i >= ny) continue;
      const int dy = y - __ldg(oy + i);
      if (dy < 0 || dy >= th) continue;
      const float wyv = __ldg(wy + dy);
      for (int b = 0; b < nj; ++b) {
        const int j = j0 + b;
        if (j < 0 || j >= nx) continue;
        const int dx = x - __ldg(ox + j);
        if (dx < 0 || dx >= tw) continue;
        const float w = __fmul_rn(wyv, __ldg(wx + dx));
        const float* p = tiles + ((long long)(i * nx + j) * K) * plane + (long long)dy * tw + dx;
#pragma unroll
        for (int k = 0; k < KB; ++k)
          if (k < K) num[k] = __fadd_rn(num[k], __fmul_rn(w, __ldcs(p + k * plane)));
        den = __fadd_rn(den, w);
      }
    }
    const long long pix = (long long)y * W + x;
    uint8_t label = 0;
    float best = 0.f;
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      if (k < K) {
        const float v = __fdiv_rn(num[k], den);
        if (out) out[k * HW + pix] = v;
        if (K == 1) label = v > threshold;
        else if (k == 0 || v > best) {      // strict: ties keep the lowest class index, as torch.argmax
          best = v;
          label = (uint8_t)k;
        }
      }
    }
    labels[pix] = label;
  }
}

template <int KB>
int launch_blend(const float* tiles, int K, int H, int W, const int* oy, const int* ox, int ny, int nx, int th, int tw,
                 const int* rf, const int* rc, const int* cf, const int* cc, const float* wy, const float* wx,
                 float threshold, float* out, uint8_t* labels, cudaStream_t st) {
  const long segs = (long)H * ((W + kThreads - 1) / kThreads);
  tile_blend_kernel<KB><<<grid_for(segs, 1), kThreads, 0, st>>>(tiles, K, H, W, oy, ox, ny, nx, th, tw, rf, rc, cf, cc,
                                                                wy, wx, threshold, out, labels);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

}  // namespace

extern "C" int rbu_tile_gather(const float* x, int nc, int H, int W, const int* oy, const int* ox, int ny, int nx,
                               int th, int tw, int t0, int Tb, float* out, void* stream) {
  RBU_CHECK_ARG(x && oy && ox && out && nc > 0 && H > 0 && W > 0 && ny > 0 && nx > 0 && th > 0 && tw > 0,
                "rbu_tile_gather: bad arguments");
  RBU_CHECK_ARG(th <= 2 * H - 1 && tw <= 2 * W - 1,
                "rbu_tile_gather: a %dx%d tile reaches beyond one reflection of a %dx%d scene", th, tw, H, W);
  RBU_CHECK_ARG(t0 >= 0 && Tb > 0 && (long long)t0 + Tb <= (long long)ny * nx,
                "rbu_tile_gather: tiles [%d, %d) outside the %d x %d tile grid", t0, t0 + Tb, ny, nx);
  const long long rows = (long long)Tb * nc * th;
  RBU_CHECK_ARG(rows < (1LL << 31), "rbu_tile_gather: %lld tile rows per call (at most 2^31 - 1)", rows);
  tile_gather_kernel<<<grid_for(rows, kThreads / 32), kThreads, 0, (cudaStream_t)stream>>>(x, nc, H, W, oy, ox, nx, th,
                                                                                           tw, t0, (int)rows, out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_tile_blend(const float* tiles, int K, int H, int W, const int* oy, const int* ox, int ny, int nx,
                              int th, int tw, const int* row_first, const int* row_count, const int* col_first,
                              const int* col_count, const float* wy, const float* wx, float threshold, float* out,
                              uint8_t* labels, void* stream) {
  RBU_CHECK_ARG(tiles && oy && ox && row_first && row_count && col_first && col_count && wy && wx && labels,
                "rbu_tile_blend: null pointer");
  RBU_CHECK_ARG(H > 0 && W > 0 && ny > 0 && nx > 0 && th > 0 && tw > 0 && (long long)ny * nx < (1LL << 31) &&
                    (long long)H * ((W + kThreads - 1) / kThreads) < (1LL << 31),
                "rbu_tile_blend: bad sizes");
  RBU_CHECK_ARG(K >= 1 && K <= kMaxK, "rbu_tile_blend: K must be in [1, %d], got %d", kMaxK, K);
  cudaStream_t st = (cudaStream_t)stream;
#define RBU_BLEND(KB) \
  launch_blend<KB>(tiles, K, H, W, oy, ox, ny, nx, th, tw, row_first, row_count, col_first, col_count, wy, wx, \
                   threshold, out, labels, st)
  if (K == 1) return RBU_BLEND(1);
  if (K == 2) return RBU_BLEND(2);
  if (K <= 4) return RBU_BLEND(4);
  if (K <= 8) return RBU_BLEND(8);
  if (K <= 16) return RBU_BLEND(16);
  return RBU_BLEND(32);
#undef RBU_BLEND
}
