// K1 / K10: implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulators in
// TMEM), operands staged by TMA as SWIZZLE_128B tiles of NHWC bf16 activations and packed bf16 weights.
//
//   D[pixel, n] = sum_{segment} sum_{tap} sum_{c}  X_seg[pixel + tap, c] * W_seg[n, tap, c]
//
// One kernel serves: 3x3 convs with dilation 1/2/4 (padding == dilation comes from TMA out-of-bounds
// zero fill), 1x1 convs, ConvTranspose2d(2, s=2) forward (GEMM with N = 4*Cout + pixel-shuffle epilogue),
// the data gradients of all of them (same kernel, re-packed weights; ConvTranspose dgrad gathers the four
// stride-2 quadrants through a 5-D tensor map) and two-segment accumulation (conv1-dgrad + shortcut-dgrad
// into one accumulator).  Replaces aten::convolution / convolution_backward(input) of
// Main_Final.py:157,159,172,126,131,205-208,261-270.
//
// Structure (persistent, warp specialised, 320 threads, 1 CTA / SM):
//   warp 0 / lane 0 : TMA producer   (A tile: 128 pixels x 64 ch, B tile: block_n x 64)   -> full[s]
//   warp 1 / lane 0 : MMA issuer     (4 x tcgen05.mma K=16 per stage, commit -> empty[s], tmem_full[a])
//   warps 2..9      : epilogue       (gemm_epilogue.cuh: tcgen05.ld 32x32b, bias/addend, bf16 pack, 16 B stores) -> tmem_empty[a]
// Two TMEM accumulator buffers let the epilogue of tile i overlap the MMAs of tile i+1.
#include "rbu_common.cuh"
#include "rbu_ptx.cuh"
#include "tma_host.cuh"
#include "gemm_epilogue.cuh"
#include <stdlib.h>

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
constexpr int NUM_THREADS = 320;   // TMA warp, MMA warp, 8 epilogue warps
constexpr int MAX_STAGES = 8;
constexpr int SMEM_LIMIT = 232448 - EPI_STAT_FLOATS * 4;  // 227 KB minus the static statistics accumulators

struct KParams {
  int N, H, W;
  int TW, TH, TN;  // conv mode: tile = TN images x TH rows x TW cols; gather mode: TH = merged (n,h) rows
  int tiles_w, tiles_h, tiles_n;
  int n_blocks, block_n, Ncols;
  int nseg;
  int taps[2], C[2], dil[2];
  int gather;
  int num_stages, tmem_cols, total_tiles;
  bf16* y;
  long long y_ld;
  int scatter, Cout;
  const float* bias;
  const float* scale;
  int relu;
  const bf16* addend;
  long long addend_ld;
  float* stats;   // [SMs][2][Ncols] (one row per CTA) column sum / sum of squares of the stored output, or NULL
  // staged epilogue (TMA stores): see the epilogue branch of the kernel
  int b_resident;         // 1: this CTA's whole weight operand (all k-blocks of its column block) is loaded once
  int tma_store;          // 1: outputs leave through the y tensor map, 0: per-thread 16-byte stores
  int log_tw, log_th;     // TW and TH are powers of two
  int Hg, Ng;             // extent of the (h, n) tile coordinates: (H, N), or (N*H, 1) for merged rows (gather)
  FastDiv fd_nb, fd_tw, fd_th, fd_cout;
};

constexpr int STG_BYTES = 32 * 64 * 2;   // one staging buffer: 32 pixels x 64 channels bf16
constexpr int BAR_BYTES = 512;           // mbarriers + TMEM slot
constexpr int ST_BUFS = 2;               // staging buffers per epilogue warp

__device__ __forceinline__ void decode_tile(const KParams& p, int tile, int& nb, int& w0, int& h0, int& n0) {
  const int sp = fast_div(tile, p.fd_nb);
  nb = tile - sp * p.n_blocks;
  const int q = fast_div(sp, p.fd_tw);
  w0 = (sp - q * p.tiles_w) * p.TW;
  const int q2 = fast_div(q, p.fd_th);
  h0 = (q - q2 * p.tiles_h) * p.TH;
  n0 = q2 * p.TN;
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmB0,
                 const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
                 const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmAd,
                 const __grid_constant__ KParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = A_BYTES + (p.b_resident ? 0 : p.block_n * 128);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.num_stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + MAX_STAGES;
  uint64_t* tfull = bars + 2 * MAX_STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* adbar = tempty + 2;            // [8 epilogue warps][3] addend-box arrival barriers
  uint64_t* bfull = adbar + 24;            // resident weight operand has landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
  uint8_t* stg_base = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(bars) + BAR_BYTES + 1023) & ~uintptr_t(1023));
  uint8_t* resb = stg_base + (p.tma_store ? 8 * ST_BUFS * STG_BYTES : 0);   // 1024-aligned: STG_BYTES is 4 KB

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  __shared__ __align__(16) float stat_smem[EPI_STAT_FLOATS];
  if (p.stats)
    for (int i = threadIdx.x; i < EPI_STAT_FLOATS; i += NUM_THREADS) stat_smem[i] = 0.f;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA0);
    ptx::prefetch_tmap(&tmB0);
    if (p.nseg > 1) {
      ptx::prefetch_tmap(&tmA1);
      ptx::prefetch_tmap(&tmB1);
    }
    if (p.tma_store) {
      ptx::prefetch_tmap(&tmY);
      if (p.addend) ptx::prefetch_tmap(&tmAd);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.num_stages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull[a], 1);
      ptx::mbar_init(&tempty[a], p.tma_store ? 4 : 8);   // staged: one half of the epilogue warps per accumulator
    }
    for (int i = 0; i < 24; ++i) ptx::mbar_init(&adbar[i], 1);
    ptx::mbar_init(bfull, 1);
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

  int kblocks_total = 0;
  for (int s = 0; s < p.nseg; ++s) kblocks_total += p.taps[s] * ((p.C[s] + BLOCK_K - 1) / BLOCK_K);

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      if (p.b_resident && blockIdx.x < p.total_tiles) {
        // every tile of this CTA has the same column block (grid % n_blocks == 0): fetch its weights once
        const int nb = blockIdx.x % p.n_blocks;
        ptx::mbar_arrive_expect_tx(bfull, (uint32_t)(kblocks_total * p.block_n * 128));
        int kb = 0;
        for (int seg = 0; seg < p.nseg; ++seg) {
          const int kch = (p.C[seg] + BLOCK_K - 1) / BLOCK_K;
          for (int tap = 0; tap < p.taps[seg]; ++tap)
            for (int kc = 0; kc < kch; ++kc, ++kb)
              ptx::tma_load_2d(resb + kb * p.block_n * 128, seg ? &tmB1 : &tmB0, bfull, tap * p.C[seg] + kc * BLOCK_K,
                               nb * p.block_n);
        }
      }
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        int nb, w0, h0, n0;
        decode_tile(p, tile, nb, w0, h0, n0);
        for (int seg = 0; seg < p.nseg; ++seg) {
          const CUtensorMap* mA = seg ? &tmA1 : &tmA0;
          const CUtensorMap* mB = seg ? &tmB1 : &tmB0;
          const int kch = (p.C[seg] + BLOCK_K - 1) / BLOCK_K;
          for (int tap = 0; tap < p.taps[seg]; ++tap) {
            int dh = 0, dw = 0;
            if (p.taps[seg] == 9) {
              dh = (tap / 3 - 1) * p.dil[seg];
              dw = (tap % 3 - 1) * p.dil[seg];
            }
            for (int kc = 0; kc < kch; ++kc) {
              ptx::mbar_wait_backoff(&empty[s], ph ^ 1);
              ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)stage_bytes);
              uint8_t* a_dst = smem + s * stage_bytes;
              uint8_t* b_dst = a_dst + A_BYTES;
              if (p.gather)
                ptx::tma_load_5d(a_dst, mA, &full[s], kc * BLOCK_K, tap & 1, w0, tap >> 1, h0);
              else
                ptx::tma_load_4d(a_dst, mA, &full[s], kc * BLOCK_K, w0 + dw, h0 + dh, n0);
              if (!p.b_resident) ptx::tma_load_2d(b_dst, mB, &full[s], tap * p.C[seg] + kc * BLOCK_K, nb * p.block_n);
              if (++s == p.num_stages) { s = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    // Whole warp walks the schedule, one elected lane issues; lean per-stage body (see conv_halo.cu).
    const uint32_t idesc = ptx::make_idesc_bf16(BLOCK_M, p.block_n, 0, 0);
    const uint32_t full_s = ptx::smem_u32(full), empty_s = ptx::smem_u32(empty);
    const uint32_t hi = ptx::desc_hi(1024);
    const uint32_t a_lo0 = ptx::desc_lo(ptx::smem_u32(smem), 16);
    const uint32_t st_step = (uint32_t)stage_bytes >> 4;
    const uint32_t rb_lo0 = ptx::desc_lo(ptx::smem_u32(resb), 16);
    const uint32_t rb_step = (uint32_t)(p.block_n * 128) >> 4;
    int s = 0, t = 0;
    uint32_t ph = 0;
    if (p.b_resident && blockIdx.x < p.total_tiles) ptx::mbar_wait(bfull, 0);
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
      const int a = t & 1;
      ptx::mbar_wait(&tempty[a], ((t >> 1) & 1) ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(a * p.block_n);
      uint32_t accumulate = 0;
      uint32_t rb_lo = rb_lo0;
      for (int seg = 0; seg < p.nseg; ++seg) {
        const int kch = (p.C[seg] + BLOCK_K - 1) / BLOCK_K;
        for (int tap = 0; tap < p.taps[seg]; ++tap) {
          for (int kc = 0; kc < kch; ++kc) {
            ptx::mbar_wait_s(full_s + s * 8, ph);
            ptx::tc_fence_after();
            const int rem = p.C[seg] - kc * BLOCK_K;
            const int ksteps = rem >= BLOCK_K ? 4 : (rem + 15) / 16;  // channels past C are TMA zero fill
            if (ptx::elect_one()) {
              const uint32_t a_lo = a_lo0 + s * st_step;
              const uint32_t b_lo = p.b_resident ? rb_lo : a_lo + (A_BYTES >> 4);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if (k < ksteps) {
                  ptx::umma_bf16(d_tmem, ptx::pack_desc(a_lo + 2 * k, hi), ptx::pack_desc(b_lo + 2 * k, hi), idesc, accumulate);
                  accumulate = 1;
                }
              }
              ptx::umma_commit_s(empty_s + s * 8);  // frees the smem stage once these MMAs retire
            }
            accumulate = 1;
            rb_lo += rb_step;
            __syncwarp();
            if (++s == p.num_stages) { s = 0; ph ^= 1; }
          }
        }
      }
      if (ptx::elect_one()) ptx::umma_commit(&tfull[a]);  // accumulator complete
      __syncwarp();
    }
  } else if (p.tma_store) {
    // ============================== epilogue, staged (warps 2..9) ==============================
    // Warp (lg, half) owns accumulator rows [32 lg, 32 lg + 32) -- 32 consecutive pixels of the tile in (n, h, w)
    // order -- of every second tile of this CTA (tiles t = half, half + 2, ...: accumulator buffer `half`), so the two
    // halves drain two tiles concurrently.  A "job" is one 64-column chunk of one tile:
    //   2 x tcgen05.ld -> scale / bias / addend / ReLU -> bf16 -> swizzled 4 KB shared-memory box -> one TMA store
    // (128-byte rows: half as many TMA row requests per byte as 32-column boxes).  Two buffers alternate; with an addend
    // its box for job k+1 is requested while job k waits for TMEM, into the buffer whose store (job k-1) has drained.
    const int ew = warp - 2;
    const int lg = warp & 3;
    const int half = ew >> 2;
    {
      uint64_t* abar = adbar + ew * 2;
      const int r2g = (lg * 32) >> p.log_tw;                       // first pixel row of the warp's group, in tile rows
      const int hg = p.gather ? r2g : (r2g & (p.TH - 1));
      const int ng = p.gather ? 0 : (r2g >> p.log_th);
      const bool has_add = p.addend != nullptr;
      uint8_t* stg = stg_base + ew * 2 * STG_BYTES;
      // 32-bit shared address of this thread's 128-byte row in buffer 0; 16-byte piece g sits at (g ^ (lane & 7)) << 4
      const uint32_t row_s = ptx::smem_u32(stg) + (uint32_t)lane * 128u;
      const uint32_t sx = (uint32_t)lane & 7u;
      const int mode = (has_add ? 1 : 0) | (p.bias ? 2 : 0) | ((p.scale || p.relu) ? 4 : 0);
      const int tstep = 2 * gridDim.x;
      const uint32_t t_lane = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(half * p.block_n);

      int tile = blockIdx.x + half * gridDim.x, c0 = 0;
      int nb = 0, w0 = 0, h0 = 0, n0 = 0;
      bool live = tile < p.total_tiles;
      if (live) decode_tile(p, tile, nb, w0, h0, n0);
      // box origin of a job in the output (or addend) tensor map
      auto box = [&](const CUtensorMap* m, bool store, uint32_t buf_s, uint64_t* bar, int jnb, int jc0, int jw0, int jh0,
                     int jn0) {
        const int col = jnb * p.block_n + jc0;
        if (p.scatter) {   // (co, j, w, i, n*H + h) view of the 2x up-sampled tensor; stores only
          const int q = fast_div(col, p.fd_cout);
          if (jh0 + hg < p.H)
            ptx::tma_store_5d_s(m, buf_s, col - q * p.Cout, q & 1, jw0, q >> 1, (jn0 + ng) * p.H + jh0 + hg);
        } else if (store) {
          ptx::tma_store_4d_s(m, buf_s, col, jw0, jh0 + hg, jn0 + ng);
        } else {
          ptx::mbar_arrive_expect_tx(bar, STG_BYTES);
          ptx::tma_load_4d_s(buf_s, m, bar, col, jw0, jh0 + hg, jn0 + ng);
        }
      };
      int b = 0, u = 0;       // staging buffer of the current job; tiles this warp has started
      uint32_t aphase = 0;
      const uint32_t stg_s = ptx::smem_u32(stg);
      // BatchNorm statistics of the stored values (p.stats): lane = channel pair of the 64-column job, which reads its two
      // channels of the warp's 32 staged pixel rows back with one conflict-free 4-byte load per row and keeps the running
      // sum / sum of squares of every job index in registers for the life of the CTA (all its tiles share one column
      // block) -- no shuffles, no exchange; the rows are flushed once at the end.
      float sacc[4][4];
#pragma unroll
      for (int J = 0; J < 4; ++J) sacc[J][0] = sacc[J][1] = sacc[J][2] = sacc[J][3] = 0.f;
      unsigned rowmask = 0;
      if (has_add && live && lane == 0) box(&tmAd, false, stg_s, &abar[0], nb, c0, w0, h0, n0);
      while (live) {
        // next job
        int tile2 = tile, c2 = c0 + 64, nb2 = nb, w2 = w0, h2 = h0, n2 = n0;
        if (c2 >= p.block_n) {
          c2 = 0;
          tile2 = tile + tstep;
          if (tile2 < p.total_tiles) decode_tile(p, tile2, nb2, w2, h2, n2);
        }
        const bool live2 = tile2 < p.total_tiles;
        if (c0 == 0) {   // first chunk of the tile: the accumulator must be complete
          ptx::mbar_wait(&tfull[half], u & 1);
          ptx::tc_fence_after();
          if (p.stats) {   // which of the warp's 32 pixel rows lie inside the tensor (conv mode only: no gather / scatter)
            const int m = lg * 32 + lane;
            const int rr = m >> p.log_tw;
            const bool inside = (w0 + (m & (p.TW - 1)) < p.W) && (h0 + (rr & (p.TH - 1)) < p.H) && (n0 + (rr >> p.log_th) < p.N);
            rowmask = __ballot_sync(0xffffffffu, inside);
          }
        }
        const bool two = c0 + 32 < p.block_n;    // false only for a 32-column GEMM
        uint32_t r[64];
        ptx::tmem_ld_32x32(t_lane + (uint32_t)c0, r);
        if (two) ptx::tmem_ld_32x32(t_lane + (uint32_t)(c0 + 32), r + 32);
        const uint32_t boff = (uint32_t)(b * STG_BYTES);
        uint4 ad[8];
        if (has_add) {
          ptx::mbar_wait(&abar[b], (aphase >> b) & 1);
          aphase ^= 1u << b;
#pragma unroll
          for (int g = 0; g < 8; ++g) ad[g] = ptx::ld_shared_v4(row_s + boff + (((uint32_t)g ^ sx) << 4));
        }
        if (lane == 0) {
          if (has_add) {
            ptx::bulk_wait_read<0>();    // the previous job's store has drained the other buffer: refill it
          } else {
            ptx::bulk_wait_read<1>();    // the store of two jobs ago has drained this buffer
          }
          if (has_add && live2) box(&tmAd, false, stg_s + (uint32_t)((b ^ 1) * STG_BYTES), &abar[b ^ 1], nb2, c2, w2, h2, n2);
        }
        ptx::tmem_ld_wait();
        if (c0 + 64 >= p.block_n) {   // accumulator drained by this warp: hand it back before the arithmetic
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&tempty[half]);
          ++u;
        }
        const int col = nb * p.block_n + c0;
        const int cb = p.scatter ? col - fast_div(col, p.fd_cout) * p.Cout : col;
        uint4 out[8];
        auto arith = [&](const uint32_t (&rr)[32], int cbh, const uint4 (&adh)[4], uint4 (&oh)[4]) {
          switch (mode) {   // warp-uniform: one lean arithmetic body per combination
            case 0: epi_math<false, false, false>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 1: epi_math<true, false, false>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 2: epi_math<false, true, false>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 3: epi_math<true, true, false>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 4: epi_math<false, false, true>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 5: epi_math<true, false, true>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            case 6: epi_math<false, true, true>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
            default: epi_math<true, true, true>(rr, p.bias, p.scale, p.relu, cbh, adh, oh); break;
          }
        };
        arith(reinterpret_cast<const uint32_t(&)[32]>(r[0]), cb, reinterpret_cast<const uint4(&)[4]>(ad[0]),
              reinterpret_cast<uint4(&)[4]>(out[0]));
        if (two)
          arith(reinterpret_cast<const uint32_t(&)[32]>(r[32]), cb + 32, reinterpret_cast<const uint4(&)[4]>(ad[4]),
                reinterpret_cast<uint4(&)[4]>(out[4]));
        __syncwarp();   // lane 0 has seen the last store from this buffer drain
#pragma unroll
        for (int g = 0; g < 8; ++g)
          if (g < 4 || two) ptx::st_shared_v4(row_s + boff + (((uint32_t)g ^ sx) << 4), out[g]);
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          box(&tmY, true, stg_s + boff, nullptr, nb, c0, w0, h0, n0);
          ptx::bulk_commit();
        }
        if (p.stats) {
          const uint32_t jb = stg_s + boff + (((uint32_t)lane & 3u) << 2);
          const uint32_t cch = (uint32_t)lane >> 2;
          float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
          for (int rr = 0; rr < 32; ++rr) {
            const uint32_t v2 = ptx::ld_shared_b32(jb + (uint32_t)rr * 128u + ((cch ^ ((uint32_t)rr & 7u)) << 4));
            if ((rowmask >> rr) & 1u) {
              const float f0 = __uint_as_float(v2 << 16), f1 = __uint_as_float(v2 & 0xffff0000u);
              s0 += f0; q0 += f0 * f0;
              s1 += f1; q1 += f1 * f1;
            }
          }
          const int jj = c0 >> 6;
#pragma unroll
          for (int J = 0; J < 4; ++J)
            if (J == jj) { sacc[J][0] += s0; sacc[J][1] += s1; sacc[J][2] += q0; sacc[J][3] += q1; }
        }
        tile = tile2; c0 = c2; nb = nb2; w0 = w2; h0 = h2; n0 = n2;
        live = live2;
        b ^= 1;
      }
      if (lane == 0) ptx::bulk_wait_read<0>();
      if (p.stats) {
        // The eight epilogue warps park their accumulators in their (drained) staging buffers -- [job][lane] x (s0, s1, q0,
        // q1) -- and after a named barrier thread (J, lane) of the first four warps adds the eight up in warp order: ONE row
        // [2][Ncols] per CTA for this CTA's column block (grid % n_blocks == 0).
        __syncwarp();                        // lane 0 has seen the last store drain this warp's buffers
#pragma unroll
        for (int J = 0; J < 4; ++J)
          ptx::st_shared_v4(stg_s + (uint32_t)((J * 32 + lane) * 16),
                            make_uint4(__float_as_uint(sacc[J][0]), __float_as_uint(sacc[J][1]), __float_as_uint(sacc[J][2]),
                                       __float_as_uint(sacc[J][3])));
        asm volatile("bar.sync 3, 256;" ::: "memory");
        const int J = ew;                    // warps 0..3 of the epilogue flush job index J = ew
        const int nbf = blockIdx.x % p.n_blocks;
        const int col = nbf * p.block_n + J * 64 + 2 * lane;
        if (J < 4 && J * 64 < p.block_n && col < p.Ncols) {
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
          const uint32_t base0 = ptx::smem_u32(stg_base) + (uint32_t)((J * 32 + lane) * 16);
          for (int w8 = 0; w8 < 8; ++w8) {
            const uint4 v = ptx::ld_shared_v4(base0 + (uint32_t)(w8 * 2 * STG_BYTES));
            a0 += __uint_as_float(v.x); a1 += __uint_as_float(v.y); a2 += __uint_as_float(v.z); a3 += __uint_as_float(v.w);
          }
          float* row_out = p.stats + (long long)blockIdx.x * 2 * p.Ncols;
          *reinterpret_cast<float2*>(row_out + col) = make_float2(a0, a1);
          *reinterpret_cast<float2*>(row_out + p.Ncols + col) = make_float2(a2, a3);
        }
      }
    }
  } else {
    // ============================== epilogue, per-thread stores (warps 2..9) ==============================
    const int lg = warp & 3;              // TMEM lane group this warp may access
    const int half = (warp - 2) >> 2;     // which of the interleaved 32-column chunks this warp drains
    const int row = lg * 32 + lane;
    EpiOut eo;
    eo.stat_acc = p.stats ? stat_smem + (warp - 2) * (EPI_STAT_CHUNKS * 64) : nullptr;
    eo.y = p.y; eo.y_ld = p.y_ld; eo.bias = p.bias; eo.scale = p.scale; eo.relu = p.relu; eo.addend = p.addend; eo.addend_ld = p.addend_ld;
    eo.Ncols = p.Ncols; eo.scatter = p.scatter; eo.Cout = p.Cout; eo.H = p.H; eo.W = p.W;
    // pixel of tile `tile` owned by this thread
    auto locate = [&](int tile, int& nb, bool& valid, long long& pix, int& n, int& h, int& w) {
      nb = tile % p.n_blocks;
      int sp = tile / p.n_blocks;
      const int w0 = (sp % p.tiles_w) * p.TW;
      sp /= p.tiles_w;
      const int h0 = (sp % p.tiles_h) * p.TH;
      const int n0 = (sp / p.tiles_h) * p.TN;
      const int wl = row % p.TW;
      const int r2 = row / p.TW;
      w = w0 + wl;
      if (p.gather) {
        const int nh = h0 + r2;
        valid = (w < p.W) && (nh < p.N * p.H);
        n = nh / p.H;
        h = nh - n * p.H;
      } else {
        h = h0 + (r2 % p.TH);
        n = n0 + r2 / p.TH;
        valid = (w < p.W) && (h < p.H) && (n < p.N);
      }
      pix = ((long long)n * p.H + h) * p.W + w;
    };
    int t = 0;
    int nb, n, h, w;
    bool valid;
    long long pix;
    uint4 ad[4];
    if (blockIdx.x < p.total_tiles) {
      locate(blockIdx.x, nb, valid, pix, n, h, w);
      epi_prefetch(eo, nb * p.block_n + half * 32, valid, pix, ad);
    }
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
      const int a = t & 1;
      const uint32_t aph = (t >> 1) & 1;
      int nb2 = 0, n2 = 0, h2 = 0, w2 = 0;
      bool valid2 = false;
      long long pix2 = 0;
      const bool more = tile + gridDim.x < p.total_tiles;
      if (more) locate(tile + gridDim.x, nb2, valid2, pix2, n2, h2, w2);
      ptx::mbar_wait(&tfull[a], aph);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(a * p.block_n);
      for (int c0 = half * 32; c0 < p.block_n; c0 += 64) {
        if (c0 != half * 32) epi_prefetch(eo, nb * p.block_n + c0, valid, pix, ad);
        epi_finish(eo, t_addr + (uint32_t)c0, nb * p.block_n + c0, valid, pix, n, h, w, ad, (c0 - half * 32) >> 6);
        if (c0 + 64 >= p.block_n && more) epi_prefetch(eo, nb2 * p.block_n + half * 32, valid2, pix2, ad);   // next tile
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[a]);
      nb = nb2; n = n2; h = h2; w = w2; valid = valid2; pix = pix2;
    }
    if (p.stats) {
      // every tile of this CTA has the same column block (grid % n_blocks == 0).  Warp (lg, half) holds chunk j = columns
      // half * 32 + 64 j; the four lane-group warps of a half are added up in lg order by warp (lg = j, half) and the CTA
      // writes ONE row.
      asm volatile("bar.sync 3, 256;" ::: "memory");
      const int nbf = blockIdx.x % p.n_blocks;
      const int j = lg;
      const int c0 = half * 32 + 64 * j;
      const int col = nbf * p.block_n + c0 + lane;
      if (c0 < p.block_n && col < p.Ncols) {
        float2 acc = make_float2(0.f, 0.f);
        for (int g4 = 0; g4 < 4; ++g4) {
          const float2 v = reinterpret_cast<const float2*>(stat_smem + (half * 4 + g4) * (EPI_STAT_CHUNKS * 64))[j * 32 + lane];
          acc.x += v.x;
          acc.y += v.y;
        }
        float* row_out = p.stats + (long long)blockIdx.x * 2 * p.Ncols;
        row_out[col] = acc.x;
        row_out[p.Ncols + col] = acc.y;
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

int pow2ceil(int v) {
  int r = 1;
  while (r < v) r <<= 1;
  return r;
}

}  // namespace

// Per-image tile statistics of the halo kernel: two 16x8-pixel half-tiles per 16x16 tile.
extern "C" int rbu_conv_tile_stats_chunks(int H, int W) { return rbu_cdiv(H, 16) * rbu_cdiv(W, 16) * 2; }
extern "C" size_t rbu_conv_tile_stats_floats(int N, int H, int W, int Ncols) {
  return (size_t)N * rbu_conv_tile_stats_chunks(H, W) * 4 * Ncols;
}

// one row [2][Ncols] per CTA (its epilogue warps' partial sums added up in warp order); rows of SMs the grid does not reach
// and columns outside a CTA's column block stay zero
extern "C" size_t rbu_conv_stats_floats(int Ncols) { return (size_t)rbu_num_sms() * 2 * Ncols; }

// BatchNorm affine from the per-(CTA, lane group) partial sums written by rbu_conv_gemm(stats != NULL):
// block = 32 channels x 32 lanes over the one-row-per-CTA partials (lane sums combined in lane order -> deterministic).
// History: 8 rows per CTA read by 8 lanes took ~39 us per BatchNorm = 0.86 ms per training step.
namespace {
constexpr int FIN_LANES = 32;
__global__ void __launch_bounds__(32 * FIN_LANES)
bn_finalize_partials_kernel(const float* __restrict__ part, int rows, int Ncols, int col_off, int C, double M, int training,
                            const float* __restrict__ gamma, const float* __restrict__ beta,
                            float* __restrict__ running_mean, float* __restrict__ running_var, float momentum, float eps,
                            float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                            float* __restrict__ rstd_out) {
  __shared__ double sh[2][FIN_LANES][32];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  double s = 0.0, q = 0.0;
  if (c < C) {
#pragma unroll 4
    for (int r = ly; r < rows; r += FIN_LANES) {
      s += (double)__ldg(part + (long)r * 2 * Ncols + col_off + c);
      q += (double)__ldg(part + (long)r * 2 * Ncols + Ncols + col_off + c);
    }
  }
  sh[0][ly][cx] = s;
  sh[1][ly][cx] = q;
  __syncthreads();
  if (ly != 0 || c >= C) return;
  double ts = 0.0, tq = 0.0;
  for (int j = 0; j < FIN_LANES; ++j) { ts += sh[0][j][cx]; tq += sh[1][j][cx]; }
  const double m = ts / M;
  double v = tq / M - m * m;
  if (v < 0.0) v = 0.0;
  const float mean = (float)m, var = (float)v;
  if (training && running_mean) {
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
    const float unbiased = M > 1.0 ? (float)(v * M / (M - 1.0)) : var;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * unbiased;
  }
  const float rstd = 1.0f / sqrtf(var + eps);
  const float sc = gamma[c] * rstd;
  scale[c] = sc;
  shift[c] = beta[c] - mean * sc;
  if (mean_out) mean_out[c] = mean;
  if (rstd_out) rstd_out[c] = rstd;
}
}  // namespace

extern "C" int rbu_bn_finalize_partials(const float* part, int Ncols, int col_off, int C, int64_t count, const float* gamma,
                                        const float* beta, float* running_mean, float* running_var, float momentum,
                                        float eps, float* scale, float* shift, float* mean_out, float* rstd_out,
                                        void* stream_) {
  RBU_CHECK_ARG(part && gamma && beta && scale && shift && Ncols > 0 && C > 0 && col_off >= 0 && col_off + C <= Ncols &&
                    count > 0, "rbu_bn_finalize_partials: bad arguments");
  bn_finalize_partials_kernel<<<rbu_cdiv(C, 32), 32 * FIN_LANES, 0, (cudaStream_t)stream_>>>(
      part, rbu_num_sms(), Ncols, col_off, C, (double)count, 1, gamma, beta, running_mean, running_var, momentum, eps,
      scale, shift, mean_out, rstd_out);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_conv_gemm(const rbu_conv_gemm_args* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  RBU_CHECK_ARG(a != nullptr, "rbu_conv_gemm: null args");
  RBU_CHECK_ARG(a->N > 0 && a->H > 0 && a->W > 0, "rbu_conv_gemm: bad pixel grid %d x %d x %d", a->N, a->H, a->W);
  RBU_CHECK_ARG(a->nseg == 1 || a->nseg == 2, "rbu_conv_gemm: nseg must be 1 or 2");
  RBU_CHECK_ARG(a->Ncols > 0 && a->Ncols % 8 == 0, "rbu_conv_gemm: Ncols=%d must be a positive multiple of 8", a->Ncols);
  RBU_CHECK_ARG(a->y != nullptr && a->y_ld % 8 == 0 && ((uintptr_t)a->y & 15) == 0,
                "rbu_conv_gemm: output view must be 16-byte aligned with ld %% 8 == 0");
  RBU_CHECK_ARG(a->bias == nullptr || ((uintptr_t)a->bias & 15) == 0, "rbu_conv_gemm: bias must be 16-byte aligned");
  RBU_CHECK_ARG(a->scale == nullptr || ((uintptr_t)a->scale & 15) == 0, "rbu_conv_gemm: scale must be 16-byte aligned");
  if (a->scatter) {
    RBU_CHECK_ARG(a->Cout > 0 && a->Ncols == 4 * a->Cout && a->Cout % 8 == 0,
                  "rbu_conv_gemm: scatter needs Ncols == 4*Cout and Cout %% 8 == 0");
    RBU_CHECK_ARG(a->addend == nullptr, "rbu_conv_gemm: addend is not supported with scatter");
  }
  // both epilogues rectify whole 8-channel groups (cb < relu per group), so only a multiple of 8 names a channel prefix
  RBU_CHECK_ARG(a->relu >= 0 && a->relu % 8 == 0 && a->relu <= (a->scatter ? a->Cout : a->Ncols),
                "rbu_conv_gemm: relu=%d must be a multiple of 8 in [0, %d]", a->relu, a->scatter ? a->Cout : a->Ncols);
  if (a->addend)
    RBU_CHECK_ARG(a->addend_ld % 8 == 0 && ((uintptr_t)a->addend & 15) == 0, "rbu_conv_gemm: addend view misaligned");
  int gather = 0;
  for (int s = 0; s < a->nseg; ++s) {
    const rbu_gemm_operand& o = a->seg[s];
    RBU_CHECK_ARG(o.x && o.w, "rbu_conv_gemm: null operand in segment %d", s);
    RBU_CHECK_ARG(o.C > 0 && o.C % 8 == 0 && o.x_ld % 8 == 0 && ((uintptr_t)o.x & 15) == 0 && ((uintptr_t)o.w & 15) == 0,
                  "rbu_conv_gemm: segment %d needs C %% 8 == 0, ld %% 8 == 0 and 16-byte aligned pointers", s);
    if (o.gather) {
      RBU_CHECK_ARG(o.taps == 4 && a->nseg == 1, "rbu_conv_gemm: gather needs taps == 4 and a single segment");
      gather = 1;
    } else {
      RBU_CHECK_ARG(o.taps == 1 || o.taps == 9, "rbu_conv_gemm: taps must be 1 or 9 (got %d)", o.taps);
      RBU_CHECK_ARG(o.taps == 1 || o.dil >= 1, "rbu_conv_gemm: dilation must be >= 1");
    }
  }

  {
    static int no_halo = -1;   // RBU_NO_HALO=1 forces the generic per-tap kernel (A/B comparisons in the tests)
    if (no_halo < 0) no_halo = getenv("RBU_NO_HALO") ? 1 : 0;
    if (!no_halo && rbu_conv_halo_supported(a)) return rbu_conv_halo_launch(a, stream);
  }
  RBU_CHECK_ARG(a->tile_stats == nullptr, "rbu_conv_gemm: tile statistics are produced by the 3x3 halo kernel only");

  KParams p;
  memset(&p, 0, sizeof(p));
  p.N = a->N; p.H = a->H; p.W = a->W;
  p.gather = gather;
  p.TW = pow2ceil(a->W) < 16 ? pow2ceil(a->W) : 16;
  if (gather) {
    p.TH = BLOCK_M / p.TW;  // merged (n,h) rows
    p.TN = 1;
    p.tiles_w = rbu_cdiv(a->W, p.TW);
    p.tiles_h = rbu_cdiv((long)a->N * a->H, p.TH);
    p.tiles_n = 1;
  } else {
    const int th_max = BLOCK_M / p.TW;
    p.TH = pow2ceil(a->H) < th_max ? pow2ceil(a->H) : th_max;
    p.TN = BLOCK_M / (p.TW * p.TH);
    p.tiles_w = rbu_cdiv(a->W, p.TW);
    p.tiles_h = rbu_cdiv(a->H, p.TH);
    p.tiles_n = rbu_cdiv(a->N, p.TN);
  }
  p.Ncols = a->Ncols;
  p.block_n = a->Ncols >= 256 ? 256 : ((a->Ncols + 31) / 32) * 32;
  p.n_blocks = rbu_cdiv(a->Ncols, p.block_n);
  p.nseg = a->nseg;
  for (int s = 0; s < a->nseg; ++s) {
    p.taps[s] = a->seg[s].taps;
    p.C[s] = a->seg[s].C;
    p.dil[s] = a->seg[s].taps == 9 ? a->seg[s].dil : 0;
  }
  p.log_tw = 0;
  while ((1 << p.log_tw) < p.TW) ++p.log_tw;
  p.log_th = 0;
  while ((1 << p.log_th) < p.TH) ++p.log_th;
  p.Hg = gather ? a->N * a->H : a->H;
  p.Ng = gather ? 1 : a->N;
  p.fd_nb = make_fastdiv(p.n_blocks);
  p.fd_tw = make_fastdiv(p.tiles_w);
  p.fd_th = make_fastdiv(p.tiles_h);
  p.fd_cout = make_fastdiv(a->scatter ? a->Cout : a->Ncols);
  // Staged epilogue (TMA stores) whenever the output is expressible as 32-pixel x 32-channel boxes of a tensor map:
  // whole 32-column chunks, and for the ConvTranspose pixel shuffle a warp's 32 pixels must be whole rows of the
  // merged (n, h) axis.  RBU_NO_TMA_STORE=1 forces the per-thread stores (A/B comparisons in the tests).
  {
    static int no_tma_store = -1;
    if (no_tma_store < 0) no_tma_store = getenv("RBU_NO_TMA_STORE") ? 1 : 0;
    const int rows = 32 / p.TW;   // rows of the h axis in one warp's box when it does not span images
    bool ok = !no_tma_store && a->Ncols % 32 == 0 && (!a->stats || (!gather && !a->scatter));
    if (a->scatter)
      ok = ok && a->Cout % 64 == 0 && ((p.TW * p.TH >= 32 && a->H % rows == 0) || p.TH == a->H);
    p.tma_store = ok ? 1 : 0;
  }
  int grid = p.tiles_w * p.tiles_h * p.tiles_n * p.n_blocks;
  if (grid > rbu_num_sms()) grid = rbu_num_sms();
  // Weights resident in shared memory when the CTA's whole operand (its column block, all k-blocks) is at most 64 KB and
  // every tile of a CTA has the same column block: the small-K GEMMs are bound by L2 -> SM traffic, of which the per-tile
  // weight reload is 17-40%.  RBU_NO_RESIDENT=1 disables.
  int kblocks_total = 0;
  for (int s = 0; s < a->nseg; ++s) kblocks_total += a->seg[s].taps * rbu_cdiv(a->seg[s].C, BLOCK_K);
  const int resb_bytes = kblocks_total * p.block_n * 128;
  {
    static int no_res = -1;
    if (no_res < 0) no_res = getenv("RBU_NO_RESIDENT") ? 1 : 0;
    p.b_resident = (!no_res && resb_bytes <= 65536 && grid % p.n_blocks == 0) ? 1 : 0;
  }
  const int staging = 1024 + (p.tma_store ? 8 * ST_BUFS * STG_BYTES : 0) + (p.b_resident ? resb_bytes : 0);
  const int stage_bytes = A_BYTES + (p.b_resident ? 0 : p.block_n * 128);
  p.num_stages = (SMEM_LIMIT - 1024 - BAR_BYTES - staging) / stage_bytes;
  if (p.num_stages > MAX_STAGES) p.num_stages = MAX_STAGES;
  p.tmem_cols = 32;
  while (p.tmem_cols < 2 * p.block_n) p.tmem_cols <<= 1;
  p.total_tiles = p.tiles_w * p.tiles_h * p.tiles_n * p.n_blocks;
  p.y = reinterpret_cast<bf16*>(a->y);
  p.y_ld = a->y_ld;
  p.scatter = a->scatter;
  p.Cout = a->scatter ? a->Cout : a->Ncols;
  p.bias = a->bias;
  p.scale = a->scale;
  p.relu = a->relu;
  p.addend = reinterpret_cast<const bf16*>(a->addend);
  p.addend_ld = a->addend_ld;
  p.stats = a->stats;

  CUtensorMap tmA[2], tmB[2];
  memset(tmA, 0, sizeof(tmA));
  memset(tmB, 0, sizeof(tmB));
  for (int s = 0; s < a->nseg; ++s) {
    const rbu_gemm_operand& o = a->seg[s];
    int rc;
    if (o.gather) {
      // x is [N, 2H, 2W, ld]; view as (C, j, w, i, n*H + h)
      const uint64_t dims[5] = {(uint64_t)o.C, 2, (uint64_t)a->W, 2, (uint64_t)a->N * a->H};
      const uint64_t str[4] = {(uint64_t)o.x_ld * 2, (uint64_t)o.x_ld * 4, (uint64_t)o.x_ld * 2 * (2 * a->W),
                               (uint64_t)o.x_ld * 4 * (2 * a->W)};
      const uint32_t box[5] = {BLOCK_K, 1, (uint32_t)p.TW, 1, (uint32_t)p.TH};
      rc = rbu_encode_tmap_bf16(&tmA[s], o.x, 5, dims, str, box);
    } else {
      const uint64_t dims[4] = {(uint64_t)o.C, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
      const uint64_t str[3] = {(uint64_t)o.x_ld * 2, (uint64_t)o.x_ld * 2 * a->W, (uint64_t)o.x_ld * 2 * a->W * a->H};
      const uint32_t box[4] = {BLOCK_K, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TN};
      rc = rbu_encode_tmap_bf16(&tmA[s], o.x, 4, dims, str, box);
    }
    if (rc) return rc;
    const uint64_t ktot = (uint64_t)o.taps * o.C;
    const uint64_t bdims[2] = {ktot, (uint64_t)a->Ncols};
    const uint64_t bstr[1] = {ktot * 2};
    const uint32_t bbox[2] = {BLOCK_K, (uint32_t)p.block_n};
    rc = rbu_encode_tmap_bf16(&tmB[s], o.w, 2, bdims, bstr, bbox);
    if (rc) return rc;
  }
  if (a->nseg == 1) {
    tmA[1] = tmA[0];
    tmB[1] = tmB[0];
  }

  // output (and addend) boxes of the staged epilogue: 64 channels x the 32 pixels of one epilogue warp, SWIZZLE_128B
  CUtensorMap tmY, tmAd;
  memset(&tmY, 0, sizeof(tmY));
  memset(&tmAd, 0, sizeof(tmAd));
  if (p.tma_store) {
    const int thb = p.TW * p.TH >= 32 ? 32 / p.TW : p.TH;    // h rows per box
    const int tnb = 32 / (p.TW * thb);                       // images per box (tiny feature maps)
    int rc;
    if (a->scatter) {
      // y is [N, 2H, 2W, ld]; view as (co, j, w, i, n*H + h)
      const uint64_t dims[5] = {(uint64_t)a->Cout, 2, (uint64_t)a->W, 2, (uint64_t)a->N * a->H};
      const uint64_t str[4] = {(uint64_t)a->y_ld * 2, (uint64_t)a->y_ld * 4, (uint64_t)a->y_ld * 2 * (2 * a->W),
                               (uint64_t)a->y_ld * 4 * (2 * a->W)};
      const uint32_t box[5] = {64, 1, (uint32_t)p.TW, 1, (uint32_t)(32 / p.TW)};
      rc = rbu_encode_tmap_bf16(&tmY, a->y, 5, dims, str, box);
    } else {
      const uint64_t dims[4] = {(uint64_t)a->Ncols, (uint64_t)a->W, (uint64_t)p.Hg, (uint64_t)p.Ng};
      const uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)thb, (uint32_t)tnb};
      const uint64_t str[3] = {(uint64_t)a->y_ld * 2, (uint64_t)a->y_ld * 2 * a->W, (uint64_t)a->y_ld * 2 * a->W * p.Hg};
      rc = rbu_encode_tmap_bf16(&tmY, a->y, 4, dims, str, box);
      if (!rc && a->addend) {
        const uint64_t astr[3] = {(uint64_t)a->addend_ld * 2, (uint64_t)a->addend_ld * 2 * a->W,
                                  (uint64_t)a->addend_ld * 2 * a->W * p.Hg};
        rc = rbu_encode_tmap_bf16(&tmAd, a->addend, 4, dims, astr, box);
      }
    }
    if (rc) return rc;
  }

  const int smem_bytes = p.num_stages * stage_bytes + 1024 + BAR_BYTES + staging;
  static std::atomic<unsigned long long> attr_set{0};      // one bit per device ordinal
  if (rbu_first_use_on_device(&attr_set))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(conv_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  if (a->stats) {
    RBU_CHECK_ARG(!a->scatter && p.block_n <= 64 * EPI_STAT_CHUNKS && grid % p.n_blocks == 0 && ((uintptr_t)a->stats & 15) == 0,
                  "rbu_conv_gemm: output statistics are not supported for this shape");
    // staged epilogue with one column block: every warp of every CTA writes its whole row, only the rows of the SMs the grid
    // does not reach need zeros
    const size_t row_floats = (size_t)2 * a->Ncols, written = (p.tma_store && p.n_blocks == 1) ? (size_t)grid : 0;
    const size_t total = rbu_conv_stats_floats(a->Ncols);
    if (written * row_floats < total)
      RBU_CHECK_CUDA(cudaMemsetAsync(a->stats + written * row_floats, 0, (total - written * row_floats) * sizeof(float), stream));
  }
  conv_gemm_kernel<<<grid, NUM_THREADS, smem_bytes, stream>>>(tmA[0], tmB[0], tmA[1], tmB[1], tmY, tmAd, p);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
