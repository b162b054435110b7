// K-class heads (1 <= K <= 32): the last 1x1 convolution of RobustUNet (`outc`, a sigmoid per class, Main_Final.py:274-277)
// and of UNet (`final`, logits, train_water_segmentation.py:246,288) for any class count, its backward, and
// nn.CrossEntropyLoss over K classes fused with per-class arg-max confusion counts (train_water_segmentation.py:304,
// 384-388).  RobustUNet at K = 1 and UNet at K = 2 keep their specialised kernels (forward_ops.cu, backward_ops.cu,
// unet_ops.cu); these serve every other class count.
#include "rbu_common.cuh"

namespace {

constexpr int KMAX = 32;

// ------------------------------------------------------------------------------------------------
// forward: one thread per pixel keeps K fp32 accumulators.  The CTA stages FT pixels x FCH channels of x in shared
// memory with coalesced 16-byte loads; the weights [K][C] sit in shared memory for the CTA's whole life.  Class planes
// are written coalesced (consecutive threads own consecutive pixels).
// ------------------------------------------------------------------------------------------------
constexpr int FT = 128;
constexpr int FCH = 64;
constexpr int FXS = FCH + 8;      // padded row: 144-byte stride keeps the per-thread 16-byte reads conflict-free

size_t fwd_smem(int KB, int C) { return (size_t)KB * C * sizeof(float) + (size_t)FT * FXS * sizeof(bf16); }

template <int KB>
__global__ void __launch_bounds__(FT)
headk_fwd_kernel(const bf16* __restrict__ x, long ld, long P, int HW, int C, int K, const float* __restrict__ w,
                 const float* __restrict__ b, int sigmoid, float* __restrict__ out, float* __restrict__ logits) {
  extern __shared__ __align__(16) unsigned char smem[];
  float* ws = reinterpret_cast<float*>(smem);                 // [KB][C], rows >= K are zero
  bf16* xs = reinterpret_cast<bf16*>(ws + KB * C);            // [FT][FXS]
  const int CH = C < FCH ? C : FCH, GCH = CH >> 3;
  for (int i = threadIdx.x; i < KB * C; i += FT) ws[i] = i < K * C ? w[i] : 0.f;
  const long ntiles = (P + FT - 1) / FT;
  for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long p0 = tile * FT, p = p0 + threadIdx.x;
    float acc[KB];
#pragma unroll
    for (int k = 0; k < KB; ++k) acc[k] = 0.f;
    for (int c0 = 0; c0 < C; c0 += CH) {
      __syncthreads();
      for (int q = threadIdx.x; q < FT * GCH; q += FT) {
        const int r = q / GCH, g = q - r * GCH;
        if (p0 + r < P) st_bf16x8(xs + r * FXS + g * 8, ld_bf16x8_stream(x + (p0 + r) * ld + c0 + g * 8));
      }
      __syncthreads();
      if (p < P)
        for (int g = 0; g < GCH; ++g) {
          float v[8];
          unpack8(*reinterpret_cast<const bf16x8*>(xs + threadIdx.x * FXS + g * 8), v);
          const float* wc = ws + c0 + g * 8;
#pragma unroll
          for (int k = 0; k < KB; ++k) {
            const float4 w0 = *reinterpret_cast<const float4*>(wc + k * C);
            const float4 w1 = *reinterpret_cast<const float4*>(wc + k * C + 4);
            float a = acc[k];
            a += w0.x * v[0]; a += w0.y * v[1]; a += w0.z * v[2]; a += w0.w * v[3];
            a += w1.x * v[4]; a += w1.y * v[5]; a += w1.z * v[6]; a += w1.w * v[7];
            acc[k] = a;
          }
        }
    }
    if (p < P) {
      const long n = p / HW, pl = p - n * HW;
      float* o = out + n * K * (long)HW + pl;
#pragma unroll
      for (int k = 0; k < KB; ++k)
        if (k < K) {
          const float z = acc[k] + __ldg(b + k);
          o[(long)k * HW] = sigmoid ? sigmoidf_acc(z) : z;
          if (logits) logits[n * K * (long)HW + pl + (long)k * HW] = z;
        }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward: per tile of TP pixels the CTA stages dz [K][TP] (fp32) and x [TP][C] (bf16) in shared memory.
//   dx: one thread per (4 pixels, 8 channels): dx = sum_k dz_k w_k, 16-byte stores;
//   dW / db: one thread per (class, 8 channels), accumulating in registers across all the CTA's tiles (db in double).
//   When K*C/8 < 256 the pairs would leave threads idle, so R = 256 / (K*C/8) groups of threads split the tile's pixels.
// Each thread group writes one partial row [K*C | K]; colsum_split sums the rows in a fixed order (no float atomics).
// ------------------------------------------------------------------------------------------------
constexpr int BT = 256;
constexpr int BPAIRS = KMAX * 32 / BT;           // (class, 8-channel group) pairs per thread at K = 32, C = 256

int bwd_tile(int C) { return C <= 128 ? 128 : 64; }
size_t bwd_smem(int K, int C) {
  const int TP = bwd_tile(C);
  return ((size_t)K * C + (size_t)K * TP) * sizeof(float) + (size_t)TP * (C + 8) * sizeof(bf16);
}
int bwd_groups(int K, int C) { return K * (C >> 3) < BT ? BT / (K * (C >> 3)) : 1; }
long bwd_blocks(int64_t P, int C) {
  const long tiles = (P + bwd_tile(C) - 1) / bwd_tile(C);
  const long cap = (long)rbu_num_sms() * 2;      // 127 registers x 256 threads: two CTAs per SM
  return tiles < cap ? (tiles < 1 ? 1 : tiles) : cap;
}

__global__ void __launch_bounds__(BT)
headk_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ probs, const bf16* __restrict__ x, long x_ld,
                 bf16* __restrict__ dx, long dx_ld, long P, int HW, int C, int K, int sigmoid, const float* __restrict__ w,
                 int TP, float* __restrict__ part, long stride) {
  extern __shared__ __align__(16) unsigned char smem[];
  float* ws = reinterpret_cast<float*>(smem);                 // [K][C]
  float* dzs = ws + K * C;                                    // [K][TP]
  bf16* xs = reinterpret_cast<bf16*>(dzs + K * TP);           // [TP][C + 8]
  const int G = C >> 3, XS = C + 8, npairs = K * G;
  const int R = npairs < BT ? BT / npairs : 1;
  for (int i = threadIdx.x; i < K * C; i += BT) ws[i] = w[i];
  float acc[BPAIRS][8];
  double accb[BPAIRS];
#pragma unroll
  for (int j = 0; j < BPAIRS; ++j) {
    accb[j] = 0.0;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[j][e] = 0.f;
  }
  const long ntiles = (P + TP - 1) / TP;
  for (long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long p0 = tile * TP;
    const int np = (int)min((long)TP, P - p0);
    __syncthreads();
    for (int i = threadIdx.x; i < K * TP; i += BT) {
      const int k = i / TP, px = i - k * TP;
      float d = 0.f;
      if (px < np) {
        const long p = p0 + px, n = p / HW;
        const long o = (n * K + k) * HW + (p - n * HW);
        d = dout[o];
        if (sigmoid) {
          const float pr = probs[o];
          d = d * pr * (1.f - pr);
        }
      }
      dzs[i] = d;
    }
    for (int q = threadIdx.x; q < np * G; q += BT) {
      const int r = q / G, g = q - r * G;
      st_bf16x8(xs + r * XS + g * 8, ld_bf16x8_stream(x + (p0 + r) * x_ld + g * 8));
    }
    __syncthreads();
    for (int q = threadIdx.x; q < (TP / 4) * G; q += BT) {
      const int px0 = (q / G) * 4, g = q % G;
      if (px0 >= np) continue;
      float o[4][8];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 8; ++e) o[j][e] = 0.f;
      for (int k = 0; k < K; ++k) {
        const float4 w0 = *reinterpret_cast<const float4*>(ws + k * C + g * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(ws + k * C + g * 8 + 4);
        const float4 d4 = *reinterpret_cast<const float4*>(dzs + k * TP + px0);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        const float dv[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 8; ++e) o[j][e] += dv[j] * wv[e];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (px0 + j < np) st_bf16x8(dx + (p0 + px0 + j) * dx_ld + g * 8, pack8(o[j]));
    }
    if (R > 1) {
      if (threadIdx.x < R * npairs) {
        const int pr = threadIdx.x % npairs, grp = threadIdx.x / npairs;
        const int k = pr / G, g = pr - k * G;
        const float* dk = dzs + k * TP;
        for (int px = grp; px < np; px += R) {
          float v[8];
          unpack8(*reinterpret_cast<const bf16x8*>(xs + px * XS + g * 8), v);
          const float d = dk[px];
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[0][e] += d * v[e];
          if (g == 0) accb[0] += d;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < BPAIRS; ++j) {
        const int pr = threadIdx.x + j * BT;
        if (pr < npairs) {
          const int k = pr / G, g = pr - k * G;
          const float* dk = dzs + k * TP;
          for (int px = 0; px < np; ++px) {
            float v[8];
            unpack8(*reinterpret_cast<const bf16x8*>(xs + px * XS + g * 8), v);
            const float d = dk[px];
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[j][e] += d * v[e];
            if (g == 0) accb[j] += d;
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < BPAIRS; ++j) {
    const int slot = threadIdx.x + j * BT;
    if (slot < R * npairs) {              // R == 1: slot is the pair; R > 1: j == 0 and slot = group * npairs + pair
      const int pr = slot % npairs, grp = slot / npairs;
      const int k = pr / G, g = pr - k * G;
      float* dst = part + ((long)blockIdx.x * R + grp) * stride;
#pragma unroll
      for (int e = 0; e < 8; ++e) dst[k * C + g * 8 + e] = acc[j][e];
      if (g == 0) dst[K * C + k] = (float)accb[j];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// nn.CrossEntropyLoss() over K classes + per-class arg-max confusion counts.  One thread per pixel reads its K logits
// (HW apart: coalesced across threads); max, log-sum-exp and the first arg-max in fp32 as ce2_partial_kernel.  Counts go
// to shared-memory integer counters (one warp-aggregated atomic per distinct counter), then one global atomic per
// (CTA, class, field).  grid (nblk, B).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cek_partial_kernel(const float* __restrict__ logits, const long long* __restrict__ target, long HW, int K,
                   float* __restrict__ partials, unsigned long long* __restrict__ counts,
                   unsigned long long* __restrict__ inv) {
  __shared__ unsigned sc[KMAX * 3];
  __shared__ float sf[8];
  __shared__ unsigned sn[8];
  for (int i = threadIdx.x; i < K * 3; i += blockDim.x) sc[i] = 0;
  __syncthreads();
  const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* z = logits + (long)b * K * HW;
  const long long* t = target + (long)b * HW;
  float loss = 0.f;
  unsigned ninv = 0;
  const long step = (long)gridDim.x * blockDim.x;
  for (long base = (long)blockIdx.x * blockDim.x; base < HW; base += step) {     // uniform trip count for the warp votes
    const long i = base + threadIdx.x;
    unsigned k1 = ~0u, k2 = ~0u;
    if (i < HW) {
      const long long y = t[i];
      float m = z[i];
      int a = 0;
      for (int k = 1; k < K; ++k) {
        const float v = z[(long)k * HW + i];
        if (v > m) { m = v; a = k; }
      }
      if (y < 0 || y >= K) {
        ++ninv;
      } else {
        float s = 0.f;
        for (int k = 0; k < K; ++k) s += expf(z[(long)k * HW + i] - m);
        loss += (m + logf(s)) - z[y * HW + i];
        if (a == (int)y) {
          k1 = a * 3;                  // TP of class a
        } else {
          k1 = a * 3 + 1;              // FP of the predicted class
          k2 = (int)y * 3 + 2;         // FN of the target class
        }
      }
    }
    const unsigned m1 = __match_any_sync(0xffffffffu, k1);
    if (k1 != ~0u && lane == __ffs(m1) - 1) atomicAdd(&sc[k1], __popc(m1));
    const unsigned m2 = __match_any_sync(0xffffffffu, k2);
    if (k2 != ~0u && lane == __ffs(m2) - 1) atomicAdd(&sc[k2], __popc(m2));
  }
  loss = warp_sum(loss);
  ninv = __reduce_add_sync(0xffffffffu, ninv);
  if (lane == 0) { sf[warp] = loss; sn[warp] = ninv; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    unsigned long long c = 0;
    for (int j = 0; j < 8; ++j) { a += sf[j]; c += sn[j]; }
    partials[(long)b * gridDim.x + blockIdx.x] = a;
    if (c) atomicAdd(&inv[b], c);
  }
  for (int i = threadIdx.x; i < K * 3; i += blockDim.x)
    if (sc[i]) atomicAdd(&counts[((long)b * K + i / 3) * 4 + i % 3], (unsigned long long)sc[i]);
}

__global__ void __launch_bounds__(256)
cek_finalize_kernel(const float* __restrict__ partials, int n, double total, long HW, int B, int K,
                    const unsigned long long* __restrict__ inv, float* __restrict__ loss_out,
                    unsigned long long* __restrict__ counts, unsigned long long* __restrict__ invalid) {
  __shared__ double sh[256];
  __shared__ unsigned long long si[256];
  double s = 0.0;
  unsigned long long c = 0;
  for (int i = threadIdx.x; i < n; i += 256) s += (double)partials[i];
  for (int i = threadIdx.x; i < B; i += 256) c += inv[i];
  sh[threadIdx.x] = s;
  si[threadIdx.x] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0;
    unsigned long long ci = 0;
    for (int j = 0; j < 256; ++j) { a += sh[j]; ci += si[j]; }
    loss_out[0] = (float)(a / total);
    invalid[0] = ci;
  }
  for (long i = threadIdx.x; i < (long)B * K; i += 256) {
    unsigned long long* q = counts + i * 4;
    q[3] = ((unsigned long long)HW - inv[i / K]) - q[0] - q[1] - q[2];
  }
}

// dlogits = (softmax - onehot) * g / (B*HW); pixels with a target outside [0, K) get 0
__global__ void __launch_bounds__(256)
cek_backward_kernel(const float* __restrict__ logits, const long long* __restrict__ target, int B, long HW, int K,
                    const float* __restrict__ gout, float* __restrict__ dlogits) {
  const float g = (gout ? gout[0] : 1.f) / ((float)B * (float)HW);
  const long total = (long)B * HW;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HW, pl = i - b * HW;
    const float* z = logits + b * K * HW + pl;
    float* d = dlogits + b * K * HW + pl;
    const long long y = target[i];
    if (y < 0 || y >= K) {
      for (int k = 0; k < K; ++k) d[(long)k * HW] = 0.f;
      continue;
    }
    float m = z[0];
    for (int k = 1; k < K; ++k) m = fmaxf(m, z[(long)k * HW]);
    float s = 0.f;
    for (int k = 0; k < K; ++k) s += expf(z[(long)k * HW] - m);
    const float inv_s = 1.f / s;
    for (int k = 0; k < K; ++k)
      d[(long)k * HW] = (expf(z[(long)k * HW] - m) * inv_s - (k == (int)y ? 1.f : 0.f)) * g;
  }
}

long cek_nblk(int64_t HW) {
  long nblk = (HW + 256 * 8 - 1) / (256 * 8);
  return nblk > 64 ? 64 : (nblk < 1 ? 1 : nblk);
}

template <int KB>
int launch_fwd(const void* x, int64_t ld, int64_t P, int HW, int C, int K, const float* w, const float* b, int sigmoid,
               float* out, float* logits, cudaStream_t st) {
  static std::atomic<unsigned long long> done{0};
  if (rbu_first_use_on_device(&done))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(headk_fwd_kernel<KB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)fwd_smem(KB, 256)));
  long blocks = (P + FT - 1) / FT;
  const long cap = (long)rbu_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  headk_fwd_kernel<KB><<<(unsigned)blocks, FT, fwd_smem(KB, C), st>>>((const bf16*)x, ld, P, HW, C, K, w, b, sigmoid, out,
                                                                      logits);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

}  // namespace

#define VIEW_OK(ptr, ld) ((ptr) != nullptr && ((uintptr_t)(ptr) & 15) == 0 && (ld) % 8 == 0)
#define HEAD_C_OK(C) ((C) >= 16 && (C) <= 256 && ((C) & ((C) - 1)) == 0)

extern "C" int rbu_headk_forward(const void* x, int64_t ld, int64_t P, int HW, int C, int K, const float* w,
                                 const float* b, int sigmoid, float* out, float* logits, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(K >= 1 && K <= KMAX, "rbu_headk_forward: K = %d classes, supported 1 <= K <= %d", K, KMAX);
  RBU_CHECK_ARG(HEAD_C_OK(C), "rbu_headk_forward: C = %d input channels, need a power of two in [16, 256]", C);
  RBU_CHECK_ARG(VIEW_OK(x, ld) && ld >= C && w && b && out && P > 0 && HW > 0 && P % HW == 0,
                "rbu_headk_forward: bad arguments");
  if (K <= 1) return launch_fwd<1>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
  if (K <= 2) return launch_fwd<2>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
  if (K <= 4) return launch_fwd<4>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
  if (K <= 8) return launch_fwd<8>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
  if (K <= 16) return launch_fwd<16>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
  return launch_fwd<32>(x, ld, P, HW, C, K, w, b, sigmoid, out, logits, st);
}

extern "C" size_t rbu_headk_backward_workspace_bytes(int64_t P, int C, int K) {
  if (!HEAD_C_OK(C) || K < 1 || K > KMAX || P <= 0) return 0;
  const long stride = (long)K * C + K;
  return ((size_t)bwd_blocks(P, C) * bwd_groups(K, C) * stride + colsum_scratch_floats((int)stride)) * sizeof(float);
}

extern "C" int rbu_headk_backward(const float* dout, const float* probs, const void* x, int64_t x_ld, void* dx,
                                  int64_t dx_ld, int64_t P, int HW, int C, int K, int sigmoid, const float* w, float* dw,
                                  float* db, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(K >= 1 && K <= KMAX, "rbu_headk_backward: K = %d classes, supported 1 <= K <= %d", K, KMAX);
  RBU_CHECK_ARG(HEAD_C_OK(C), "rbu_headk_backward: C = %d input channels, need a power of two in [16, 256]", C);
  RBU_CHECK_ARG(dout && (probs || !sigmoid) && VIEW_OK(x, x_ld) && VIEW_OK(dx, dx_ld) && x_ld >= C && dx_ld >= C && w &&
                    dw && db && P > 0 && HW > 0 && P % HW == 0,
                "rbu_headk_backward: bad arguments");
  const size_t need = rbu_headk_backward_workspace_bytes(P, C, K);
  RBU_CHECK_ARG(workspace && workspace_bytes >= need, "rbu_headk_backward: workspace too small (%zu < %zu bytes)",
                workspace_bytes, need);
  static std::atomic<unsigned long long> done{0};
  if (rbu_first_use_on_device(&done))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(headk_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)bwd_smem(KMAX, 256)));
  const int blocks = (int)bwd_blocks(P, C), rows = blocks * bwd_groups(K, C);
  const long stride = (long)K * C + K;
  float* part = (float*)workspace;
  headk_bwd_kernel<<<blocks, BT, bwd_smem(K, C), st>>>(dout, probs, (const bf16*)x, x_ld, (bf16*)dx, dx_ld, P, HW, C, K,
                                                      sigmoid, w, bwd_tile(C), part, stride);
  RBU_CHECK_LAUNCH();
  return colsum_split(part, rows, stride, K * C, dw, K, db, part + (size_t)rows * stride, st);
}

extern "C" size_t rbu_cek_workspace_bytes(int B, int64_t HW, int K) {
  (void)K;
  if (B <= 0 || HW <= 0) return 0;
  return (size_t)B * sizeof(unsigned long long) + (size_t)B * cek_nblk(HW) * sizeof(float);
}

extern "C" int rbu_cek_forward(const float* logits, const int64_t* target, int B, int64_t HW, int K, void* workspace,
                               size_t workspace_bytes, float* loss_out, int64_t* class_counts, int64_t* invalid,
                               void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  RBU_CHECK_ARG(K >= 1 && K <= KMAX, "rbu_cek_forward: K = %d classes, supported 1 <= K <= %d", K, KMAX);
  RBU_CHECK_ARG(B > 0 && B <= 65535, "rbu_cek_forward: B = %d images, supported 1 <= B <= 65535", B);
  RBU_CHECK_ARG(logits && target && loss_out && class_counts && invalid && HW > 0, "rbu_cek_forward: bad arguments");
  RBU_CHECK_ARG(workspace && ((uintptr_t)workspace & 7) == 0 && workspace_bytes >= rbu_cek_workspace_bytes(B, HW, K),
                "rbu_cek_forward: workspace too small or misaligned");
  const long nblk = cek_nblk(HW);
  unsigned long long* inv = (unsigned long long*)workspace;
  float* partials = (float*)(inv + B);
  RBU_CHECK_CUDA(cudaMemsetAsync(class_counts, 0, (size_t)B * K * 4 * sizeof(int64_t), st));
  RBU_CHECK_CUDA(cudaMemsetAsync(inv, 0, (size_t)B * sizeof(unsigned long long), st));
  cek_partial_kernel<<<dim3((unsigned)nblk, B), 256, 0, st>>>(logits, (const long long*)target, HW, K, partials,
                                                              (unsigned long long*)class_counts, inv);
  RBU_CHECK_LAUNCH();
  cek_finalize_kernel<<<1, 256, 0, st>>>(partials, (int)(B * nblk), (double)B * (double)HW, HW, B, K, inv, loss_out,
                                         (unsigned long long*)class_counts, (unsigned long long*)invalid);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_cek_backward(const float* logits, const int64_t* target, int B, int64_t HW, int K,
                                const float* grad_out, float* dlogits, void* stream_) {
  RBU_CHECK_ARG(K >= 1 && K <= KMAX, "rbu_cek_backward: K = %d classes, supported 1 <= K <= %d", K, KMAX);
  RBU_CHECK_ARG(logits && target && dlogits && B > 0 && B <= 65535 && HW > 0, "rbu_cek_backward: bad arguments");
  const long total = (long)B * HW;
  long blocks = (total + 255) / 256;
  const long cap = (long)rbu_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  cek_backward_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(logits, (const long long*)target, B, HW, K,
                                                                           grad_out, dlogits);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
