// K11: weight-gradient implicit GEMM on tcgen05 tensor cores.
//
//   R[m][t][n] = sum over pixels p of  A[p, m] * B[p (+) tap t, n]
//
// conv:            A = dy (M = Cout), B = x shifted by the 3x3 tap (dilation d) or unshifted (1x1), N = Cin
// ConvTranspose2d: A = x  (M = Cin),  B = dout gathered at quadrant (i,j) = tap,                    N = Cout
// The reduction dimension is the pixel index, so both operands are "MN-major" for the MMA: the TMA boxes
// (rows = pixels, 128 B = 64 channels, SWIZZLE_128B) are exactly the canonical MN-major layout and are shared
// with the forward kernel's activation tensor maps.  Split-K over pixel tiles with fp32 partials in a
// caller-provided workspace and an ordered reduction (deterministic; no float atomics) that writes the
// gradient in torch layout  out[(m*Ntot + n)*taps + t]  (Conv2d [Cout,Cin,kh,kw], ConvTranspose2d [Cin,Cout,2,2]).
// Replaces aten::convolution_backward(weight) of Main_Final.py:157,159,172,126,131,205-208,261-270.
//
// Work item = (M block, N block, tap group of T taps, pixel-tile range).  Two TMA rings: the A tile is loaded
// once per pixel tile and reused for the T taps; B tiles stream per tap.  T accumulators live in TMEM.
#include "rbu_common.cuh"
#include "rbu_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int TILE_PX = 128;
constexpr int BOX_BYTES = TILE_PX * 128;  // one 64-channel box: 16 KB
constexpr int NUM_THREADS = 192;
constexpr int A_STAGES = 2;
constexpr int SMEM_LIMIT = 232448;

struct WParams {
  int N, H, W;
  int TW, TH, TN;
  int tiles_w, tiles_h, tiles_n, tiles_total;
  int Mtot, Ntot, taps, dil, gather;
  int BM, BN, T;                 // block sizes; T taps per work item
  int m_blocks, n_blocks, t_groups, ksplit, items;
  int b_stages, tmem_cols;
  float* partial;                // [ksplit][Mtot][taps][Ntot]
};

__device__ __forceinline__ void decode_item(const WParams& p, int item, int& mb, int& nb, int& tg, int& ks) {
  mb = item % p.m_blocks; item /= p.m_blocks;
  nb = item % p.n_blocks; item /= p.n_blocks;
  tg = item % p.t_groups;
  ks = item / p.t_groups;
}
__device__ __forceinline__ void tile_origin(const WParams& p, int tile, int& w0, int& h0, int& n0) {
  w0 = (tile % p.tiles_w) * p.TW;
  tile /= p.tiles_w;
  h0 = (tile % p.tiles_h) * p.TH;
  n0 = (tile / p.tiles_h) * p.TN;
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ WParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int a_boxes = p.BM / 64 > 0 ? (p.BM + 63) / 64 : 1;
  const int b_boxes = (p.BN + 63) / 64;
  const int a_bytes = a_boxes * BOX_BYTES;
  const int b_bytes = b_boxes * BOX_BYTES;
  uint8_t* smA = smem;
  uint8_t* smB = smem + A_STAGES * a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smB + p.b_stages * b_bytes);
  uint64_t* fullA = bars;            // [A_STAGES]
  uint64_t* emptyA = bars + 2;       // [A_STAGES]
  uint64_t* fullB = bars + 4;        // [8]
  uint64_t* emptyB = bars + 12;      // [8]
  uint64_t* tfull = bars + 20;
  uint64_t* tempty = bars + 21;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < A_STAGES; ++s) { ptx::mbar_init(&fullA[s], 1); ptx::mbar_init(&emptyA[s], 1); }
    for (int s = 0; s < p.b_stages; ++s) { ptx::mbar_init(&fullB[s], 1); ptx::mbar_init(&emptyB[s], 1); }
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, 4);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
        int mb, nb, tg, ks;
        decode_item(p, item, mb, nb, tg, ks);
        const int t_begin = tg * p.T;
        const int t_end = min(t_begin + p.T, p.taps);
        const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
        const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
        for (int tile = tile0; tile < tile1; ++tile) {
          int w0, h0, n0;
          tile_origin(p, tile, w0, h0, n0);
          {
            const int s = sa;
            const uint32_t ph = pha;
            if (++sa == A_STAGES) { sa = 0; pha ^= 1; }
            ptx::mbar_wait(&emptyA[s], ph ^ 1);
            ptx::mbar_arrive_expect_tx(&fullA[s], (uint32_t)a_bytes);
            for (int bx = 0; bx < a_boxes; ++bx)
              ptx::tma_load_4d(smA + s * a_bytes + bx * BOX_BYTES, &tmA, &fullA[s], mb * p.BM + bx * 64, w0, h0, n0);
          }
          for (int t = t_begin; t < t_end; ++t) {
            const int s = sb;
            const uint32_t ph = phb;
            if (++sb == p.b_stages) { sb = 0; phb ^= 1; }
            ptx::mbar_wait(&emptyB[s], ph ^ 1);
            ptx::mbar_arrive_expect_tx(&fullB[s], (uint32_t)b_bytes);
            for (int bx = 0; bx < b_boxes; ++bx) {
              uint8_t* dst = smB + s * b_bytes + bx * BOX_BYTES;
              const int c0 = nb * p.BN + bx * 64;
              if (p.gather) {
                ptx::tma_load_5d(dst, &tmB, &fullB[s], c0, t & 1, w0, t >> 1, h0);
              } else {
                int dh = 0, dw = 0;
                if (p.taps == 9) { dh = (t / 3 - 1) * p.dil; dw = (t % 3 - 1) * p.dil; }
                ptx::tma_load_4d(dst, &tmB, &fullB[s], c0, w0 + dw, h0 + dh, n0);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // MMA issuer: the whole warp walks the schedule (uniform control flow), one elected lane issues; descriptor
    // halves are precomputed and the ring indices wrap by compare (the issuing thread must stay well below the
    // 8 x 64-cycle MMA time of a tap).
    const uint32_t idesc = ptx::make_idesc_bf16(p.BM, p.BN, 1, 1);
    const uint32_t fullA_s = ptx::smem_u32(fullA), emptyA_s = ptx::smem_u32(emptyA);
    const uint32_t fullB_s = ptx::smem_u32(fullB), emptyB_s = ptx::smem_u32(emptyB);
    const uint32_t hi = ptx::desc_hi(1024);
    const uint32_t a_lo0 = ptx::desc_lo(ptx::smem_u32(smA), BOX_BYTES), b_lo0 = ptx::desc_lo(ptx::smem_u32(smB), BOX_BYTES);
    const uint32_t a_step = (uint32_t)a_bytes >> 4, b_step = (uint32_t)b_bytes >> 4;
    int sa = 0, sb = 0, it = 0;
    uint32_t pha = 0, phb = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int mb, nb, tg, ks;
      decode_item(p, item, mb, nb, tg, ks);
      const int ntap = min(tg * p.T + p.T, p.taps) - tg * p.T;
      const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
      const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
      ptx::mbar_wait(tempty, (it & 1) ^ 1);
      ptx::tc_fence_after();
      uint32_t accumulate = 0;
      for (int tile = tile0; tile < tile1; ++tile) {
        ptx::mbar_wait_s(fullA_s + sa * 8, pha);
        ptx::tc_fence_after();
        const uint32_t a_lo = a_lo0 + sa * a_step;
        for (int t = 0; t < ntap; ++t) {
          ptx::mbar_wait_s(fullB_s + sb * 8, phb);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t b_lo = b_lo0 + sb * b_step;
            const uint32_t d_tmem = tmem_base + (uint32_t)(t * p.BN);
#pragma unroll
            for (int k = 0; k < TILE_PX / 16; ++k)
              ptx::umma_bf16(d_tmem, ptx::pack_desc(a_lo + k * (2048 >> 4), hi), ptx::pack_desc(b_lo + k * (2048 >> 4), hi),
                             idesc, (k > 0) ? 1u : accumulate);
            ptx::umma_commit_s(emptyB_s + sb * 8);
          }
          __syncwarp();
          if (++sb == p.b_stages) { sb = 0; phb ^= 1; }
        }
        accumulate = 1;
        if (ptx::elect_one()) ptx::umma_commit_s(emptyA_s + sa * 8);
        __syncwarp();
        if (++sa == A_STAGES) { sa = 0; pha ^= 1; }
      }
      if (ptx::elect_one()) ptx::umma_commit(tfull);
      __syncwarp();
    }
  } else {
    const int lg = warp & 3;
    int it = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int mb, nb, tg, ks;
      decode_item(p, item, mb, nb, tg, ks);
      const int t_begin = tg * p.T;
      const int t_end = min(t_begin + p.T, p.taps);
      // accumulator row owned by this thread (M=128: lane == row; M=64: rows 16*lg + lane in lanes 0..15)
      int m_local;
      bool row_ok;
      if (p.BM == 128) { m_local = lg * 32 + lane; row_ok = true; }
      else { m_local = lg * 16 + lane; row_ok = lane < 16; }
      const int m = mb * p.BM + m_local;
      row_ok = row_ok && (m < p.Mtot);
      ptx::mbar_wait(tfull, it & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
      for (int t = t_begin; t < t_end; ++t) {
        for (int c0 = 0; c0 < p.BN; c0 += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32(t_addr + (uint32_t)((t - t_begin) * p.BN + c0), r);
          ptx::tmem_ld_wait();
          const int n0 = nb * p.BN + c0;
          if (row_ok && n0 < p.Ntot) {
            float* dst = p.partial + (((long)ks * p.Mtot + m) * p.taps + t) * p.Ntot + n0;
            if (n0 + 32 <= p.Ntot && (p.Ntot & 3) == 0) {
#pragma unroll
              for (int g = 0; g < 8; ++g)
                *reinterpret_cast<float4*>(dst + g * 4) = make_float4(__uint_as_float(r[g * 4]), __uint_as_float(r[g * 4 + 1]),
                                                                      __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
            } else {
              for (int e = 0; e < 32; ++e)
                if (n0 + e < p.Ntot) dst[e] = __uint_as_float(r[e]);
            }
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// out[(m*Ntot + n)*taps + t] = sum_ks partial[ks][m][t][n]     (fixed order; fp32)
// Block = one output row m and a run of NCH columns: 256 threads = NCH columns x KL split-K lanes.  Lane j adds the
// partials k = j, j + KL, ... (four independent accumulators, fixed assignment), the KL lane sums are combined in lane
// order through shared memory, and the NCH x taps results -- contiguous in the torch layout -- leave as one coalesced
// run.  (The element-per-thread version walked the whole split-K chain in one thread -- 63 us for a 2048-element
// gradient with 148 partials -- and wrote with a stride of `taps` floats.)
template <int NCH>
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, int ksplit, int Mtot, int taps, int Ntot,
                    float* __restrict__ out, int accumulate) {
  constexpr int KL = 256 / NCH;
  constexpr int MAXT = 9;
  __shared__ float lane_sum[KL][MAXT][NCH + 1];
  __shared__ float res[NCH * MAXT];
  const int nchunks = (Ntot + NCH - 1) / NCH;
  const int m = blockIdx.x / nchunks, n0 = (blockIdx.x - m * nchunks) * NCH;
  const int nn = threadIdx.x % NCH, kl = threadIdx.x / NCH;
  const int n = n0 + nn;
  const long total = (long)Mtot * taps * Ntot;
  // all taps of this thread's column at once: the loads of the whole (tap, k) set are independent
  float acc[MAXT][2];
#pragma unroll
  for (int t = 0; t < MAXT; ++t) acc[t][0] = acc[t][1] = 0.f;
  if (n < Ntot) {
    const float* src = partial + (long)m * taps * Ntot + n;
    int k = kl;
    for (; k + KL < ksplit; k += 2 * KL) {
#pragma unroll
      for (int t = 0; t < MAXT; ++t)
        if (t < taps) {
          acc[t][0] += __ldg(src + (long)k * total + (long)t * Ntot);
          acc[t][1] += __ldg(src + (long)(k + KL) * total + (long)t * Ntot);
        }
    }
    if (k < ksplit) {   // 32-bit tap offsets: with 64-bit ones ptxas spills a register pair around this tail
#pragma unroll
      for (int t = 0; t < MAXT; ++t)
        if (t < taps) acc[t][0] += __ldg(src + (long)k * total + t * Ntot);
    }
  }
#pragma unroll
  for (int t = 0; t < MAXT; ++t)
    if (t < taps) lane_sum[kl][t][nn] = acc[t][0] + acc[t][1];
  __syncthreads();
  for (int i = threadIdx.x; i < NCH * taps; i += 256) {
    const int t = i / NCH, c = i - t * NCH;
    float sum = lane_sum[0][t][c];
    for (int j = 1; j < KL; ++j) sum += lane_sum[j][t][c];
    res[c * taps + t] = sum;
  }
  __syncthreads();
  const int nw = min(NCH, Ntot - n0);
  float* o = out + ((long)m * Ntot + n0) * taps;
  for (int i = threadIdx.x; i < nw * taps; i += 256) o[i] = accumulate ? o[i] + res[i] : res[i];
}

int pow2ceil_w(int v) {
  int r = 1;
  while (r < v) r <<= 1;
  return r;
}

struct Plan {
  WParams p;
  size_t ws_bytes;
};

int make_plan(const rbu_wgrad_args* a, Plan* pl) {
  WParams& p = pl->p;
  memset(&p, 0, sizeof(p));
  p.N = a->N; p.H = a->H; p.W = a->W;
  p.gather = a->gather;
  p.taps = a->taps;
  p.dil = a->taps == 9 ? a->dil : 0;
  p.Mtot = a->Ca;
  p.Ntot = a->Cb;
  p.TW = pow2ceil_w(a->W) < 16 ? pow2ceil_w(a->W) : 16;
  if (a->gather) {
    p.TH = TILE_PX / p.TW;
    p.TN = 1;
    p.tiles_w = rbu_cdiv(a->W, p.TW);
    p.tiles_h = rbu_cdiv((long)a->N * a->H, p.TH);
    p.tiles_n = 1;
  } else {
    const int th_max = TILE_PX / p.TW;
    p.TH = pow2ceil_w(a->H) < th_max ? pow2ceil_w(a->H) : th_max;
    p.TN = TILE_PX / (p.TW * p.TH);
    p.tiles_w = rbu_cdiv(a->W, p.TW);
    p.tiles_h = rbu_cdiv(a->H, p.TH);
    p.tiles_n = rbu_cdiv(a->N, p.TN);
  }
  p.tiles_total = p.tiles_w * p.tiles_h * p.tiles_n;
  p.BM = a->Ca > 64 ? 128 : 64;
  p.BN = a->Cb > 64 ? 128 : 64;
  p.T = a->taps == 9 ? 3 : a->taps;   // 3 x 128 or 4 x 128 columns fit the 512-column TMEM
  p.m_blocks = rbu_cdiv(a->Ca, p.BM);
  p.n_blocks = rbu_cdiv(a->Cb, p.BN);
  p.t_groups = rbu_cdiv(a->taps, p.T);
  const int base_items = p.m_blocks * p.n_blocks * p.t_groups;
  int ks = rbu_cdiv(2L * rbu_num_sms(), base_items);
  if (ks > p.tiles_total) ks = p.tiles_total;
  if (ks < 1) ks = 1;
  p.ksplit = ks;
  p.items = base_items * ks;
  const int a_bytes = ((p.BM + 63) / 64) * BOX_BYTES, b_bytes = ((p.BN + 63) / 64) * BOX_BYTES;
  p.b_stages = (SMEM_LIMIT - 2048 - A_STAGES * a_bytes) / b_bytes;
  if (p.b_stages > 8) p.b_stages = 8;
  p.tmem_cols = 32;
  while (p.tmem_cols < p.T * p.BN) p.tmem_cols <<= 1;
  pl->ws_bytes = (size_t)ks * a->Ca * a->taps * a->Cb * sizeof(float);
  return 0;
}

int check_args(const rbu_wgrad_args* a) {
  RBU_CHECK_ARG(a != nullptr, "rbu_wgrad_gemm: null args");
  RBU_CHECK_ARG(a->N > 0 && a->H > 0 && a->W > 0, "rbu_wgrad_gemm: bad pixel grid");
  RBU_CHECK_ARG(a->Ca > 0 && a->Ca % 8 == 0 && a->Cb > 0 && a->Cb % 8 == 0, "rbu_wgrad_gemm: channel counts must be multiples of 8");
  RBU_CHECK_ARG(a->a_ld % 8 == 0 && a->b_ld % 8 == 0, "rbu_wgrad_gemm: ld must be a multiple of 8");
  if (a->gather) RBU_CHECK_ARG(a->taps == 4, "rbu_wgrad_gemm: gather needs taps == 4");
  else RBU_CHECK_ARG(a->taps == 1 || (a->taps == 9 && a->dil >= 1), "rbu_wgrad_gemm: taps must be 1 or 9 (dil >= 1)");
  return RBU_OK;
}

}  // namespace

void rbu_wgrad_reduce_launch(const float* partial, int ksplit, int Mtot, int taps, int Ntot, float* out, int accumulate,
                             cudaStream_t stream) {
  // 64-column runs (4 split-K lanes) for wide gradients, 32 / 16 columns (8 / 16 lanes) for narrow ones with long chains
  if (Ntot >= 64 && ksplit <= 16)
    wgrad_reduce_kernel<64><<<Mtot * ((Ntot + 63) / 64), 256, 0, stream>>>(partial, ksplit, Mtot, taps, Ntot, out, accumulate);
  else if (Ntot >= 32 && ksplit <= 64)
    wgrad_reduce_kernel<32><<<Mtot * ((Ntot + 31) / 32), 256, 0, stream>>>(partial, ksplit, Mtot, taps, Ntot, out, accumulate);
  else
    wgrad_reduce_kernel<16><<<Mtot * ((Ntot + 15) / 16), 256, 0, stream>>>(partial, ksplit, Mtot, taps, Ntot, out, accumulate);
}

extern "C" size_t rbu_wgrad_workspace_bytes(const rbu_wgrad_args* a) {
  if (check_args(a) != RBU_OK) return 0;
  if (rbu_wgrad_halo_supported(a)) return rbu_wgrad_halo_workspace_bytes(a);
  Plan pl;
  make_plan(a, &pl);
  return pl.ws_bytes;
}

static int rbu_wgrad_generic_launch(const rbu_wgrad_args* a, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc;
  Plan pl;
  make_plan(a, &pl);
  WParams& p = pl.p;
  RBU_CHECK_ARG(workspace && workspace_bytes >= pl.ws_bytes && ((uintptr_t)workspace & 15) == 0,
                "rbu_wgrad_gemm: workspace too small (%zu < %zu)", workspace_bytes, pl.ws_bytes);
  p.partial = reinterpret_cast<float*>(workspace);

  CUtensorMap tmA, tmB;
  {
    // A: unshifted operand on the (N,H,W) grid
    uint64_t dims[4], str[3];
    uint32_t box[4];
    dims[0] = (uint64_t)a->Ca;
    str[0] = (uint64_t)a->a_ld * 2;
    dims[1] = (uint64_t)a->W;
    box[0] = 64; box[1] = (uint32_t)p.TW; box[2] = (uint32_t)p.TH; box[3] = (uint32_t)p.TN;
    if (a->gather) {
      dims[2] = (uint64_t)a->N * a->H; dims[3] = 1;
      str[1] = (uint64_t)a->a_ld * 2 * a->W;
      str[2] = str[1] * dims[2];
    } else {
      dims[2] = (uint64_t)a->H; dims[3] = (uint64_t)a->N;
      str[1] = (uint64_t)a->a_ld * 2 * a->W;
      str[2] = str[1] * a->H;
    }
    rc = rbu_encode_tmap_bf16(&tmA, a->a, 4, dims, str, box);
    if (rc) return rc;
  }
  if (a->gather) {
    const uint64_t dims[5] = {(uint64_t)a->Cb, 2, (uint64_t)a->W, 2, (uint64_t)a->N * a->H};
    const uint64_t str[4] = {(uint64_t)a->b_ld * 2, (uint64_t)a->b_ld * 4, (uint64_t)a->b_ld * 2 * (2 * a->W),
                             (uint64_t)a->b_ld * 4 * (2 * a->W)};
    const uint32_t box[5] = {64, 1, (uint32_t)p.TW, 1, (uint32_t)p.TH};
    rc = rbu_encode_tmap_bf16(&tmB, a->b, 5, dims, str, box);
  } else {
    const uint64_t dims[4] = {(uint64_t)a->Cb, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->b_ld * 2, (uint64_t)a->b_ld * 2 * a->W, (uint64_t)a->b_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TN};
    rc = rbu_encode_tmap_bf16(&tmB, a->b, 4, dims, str, box);
  }
  if (rc) return rc;

  const int a_bytes = ((p.BM + 63) / 64) * BOX_BYTES, b_bytes = ((p.BN + 63) / 64) * BOX_BYTES;
  const int smem_bytes = A_STAGES * a_bytes + p.b_stages * b_bytes + 1024 + 256;
  static std::atomic<unsigned long long> attr_set{0};      // one bit per device ordinal
  if (rbu_first_use_on_device(&attr_set))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(wgrad_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  const int grid = p.items < rbu_num_sms() ? p.items : rbu_num_sms();
  wgrad_gemm_kernel<<<grid, NUM_THREADS, smem_bytes, stream>>>(tmA, tmB, p);
  RBU_CHECK_LAUNCH();
  rbu_wgrad_reduce_launch(p.partial, p.ksplit, p.Mtot, p.taps, p.Ntot, a->out, a->accumulate, stream);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_wgrad_gemm(const rbu_wgrad_args* a, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  int rc = check_args(a);
  if (rc) return rc;
  RBU_CHECK_ARG(a->a && a->b && a->out && ((uintptr_t)a->a & 15) == 0 && ((uintptr_t)a->b & 15) == 0,
                "rbu_wgrad_gemm: null or misaligned pointer");
  if (rbu_wgrad_halo_supported(a)) {
    RBU_CHECK_ARG(workspace && workspace_bytes >= rbu_wgrad_halo_workspace_bytes(a) && ((uintptr_t)workspace & 15) == 0,
                  "rbu_wgrad_gemm: workspace too small");
    return rbu_wgrad_halo_launch(a, workspace, stream);
  }
  return rbu_wgrad_generic_launch(a, workspace, workspace_bytes, stream);
}
