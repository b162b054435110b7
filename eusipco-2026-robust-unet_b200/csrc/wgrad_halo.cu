// K11, halo variant: weight gradient of a 3x3 (dilation 1) convolution on tcgen05 tensor cores with ALL NINE TAPS
// accumulated from ONE activation tile.
//
//   dW[cout][cin][tap] = sum over pixels p of  dy[p, cout] * x[p (+) tap, cin]
//
// The generic kernel (wgrad_gemm.cu) streams one shifted x tile per tap and, for 64-channel layers, runs M = 64 MMAs
// (half rate): 280-460 TFLOP/s on the 64-channel level, 750-850 elsewhere (L2->SM traffic bound, 98 FLOP/B).
// Here a work item is (64 input channels) x (64 output channels) x (a range of 8x16-pixel tiles):
//   * the x operand is the tile's 10 x 24-slot halo (18 slots used; 3072-byte row pitch), loaded by ONE TMA box and
//     reused by all 9 taps through the start address of the MN-major UMMA descriptor (same trick as conv_halo.cu);
//   * the x side is the MMA's M dimension and two taps are stacked into one M = 128 instruction: the descriptor's
//     leading-byte-offset (distance between the two 64-channel column blocks) is simply the distance between the
//     two taps' start addresses in the halo buffer -- 128 B for (dx, dx+1), 3072 B for (dy, dy+1).  Pairs
//     (0,1) (3,4) (6,7) (2,5) and the single tap 8 (M = 64) give 5 accumulators x 64 columns = 320 TMEM columns;
//   * the dy operand (N = 64) is one plain 8x16-pixel box.
// Per tile: 46 KB from L2 for 9.4 MFLOP (205 FLOP/B), 40 MMAs per barrier round trip.
// Split-K over tile ranges with fp32 partials and the ordered reduction of wgrad_gemm.cu (deterministic).
// Replaces aten::convolution_backward(weight) of Main_Final.py:157,159,205-206.
//
// Second form (wgrad_halo2_kernel, used whenever Cout is a multiple of 128): the roles of the operands are swapped.
// The form above runs M = 128 x N = 64 MMAs, which read 6 KB of operands from shared memory per 32 tensor-pipe cycles
// (192 B/clk against the 128 B/clk the SM delivers: ncu l1tex__data_pipe_tc_wavefronts_mem_shared 81 %, tensor pipe
// 50-61 %), and the 9 x 64 = 576 fp32 columns of a 64 x 64 x 9 block rule out N = 128 in the 512-column TMEM.  With
//   * dy as the M side (128 output channels = two 64-channel boxes, leading-byte-offset = one box) and
//   * the x halo as the N side, loaded with 32 channels per pixel (SWIZZLE_64B, 64-byte pixel pitch) so that the THREE
//     taps of a kernel row are three 32-channel MN-atoms 64 bytes apart: N = 96 with leading-byte-offset = 64 B,
// a work item is 128 output channels x 32 input channels x 9 taps = 3 accumulators x 96 columns (288 of 512), every MMA
// is M128 x N96 x K16 (7 KB per 48 cycles = 146 B/clk) and the L2 traffic per FLOP is unchanged (47 KB per 9.4 MFLOP).
// The epilogue thread (= output channel) reads, per tap, 32 consecutive input channels = one 128-byte run of the partials.
#include "rbu_common.cuh"
#include "rbu_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int TILE_W = 16, TILE_H = 8;
constexpr int HALO_W = 24, HALO_H = 10;
constexpr int X_BYTES = HALO_W * HALO_H * 128;   // 30720
constexpr int DY_BYTES = TILE_W * TILE_H * 128;  // 16384
constexpr int STAGE_BYTES = X_BYTES + DY_BYTES;  // 47104 (multiple of 1024)
constexpr int MAX_STAGES = 4;
constexpr int NUM_THREADS = 192;
constexpr int SMEM_LIMIT = 232448;
constexpr int NACC = 5;

struct HWParams {
  int N, H, W;
  int tiles_w, tiles_h, tiles_total;
  int Cout, Cin;
  int cin_blocks, cout_blocks, ksplit, items;
  int stages;       // smem ring depth (<= MAX_STAGES)
  int CB, OB;       // input / output channels per work item: 64 x 64 (wgrad_halo_kernel) or 32 x 128 (wgrad_halo2_kernel)
  float* partial;   // [ksplit][Cout][9][Cin]
};

__device__ __forceinline__ void decode(const HWParams& p, int item, int& cb, int& ob, int& ks) {
  cb = item % p.cin_blocks; item /= p.cin_blocks;
  ob = item % p.cout_blocks;
  ks = item / p.cout_blocks;
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                  const __grid_constant__ HWParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int stage_bytes = STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.stages * stage_bytes);
  uint64_t* full = bars;             // [MAX_STAGES]
  uint64_t* empty = bars + MAX_STAGES;   // [MAX_STAGES]
  uint64_t* tfull = bars + 2 * MAX_STAGES;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmX);
    ptx::prefetch_tmap(&tmDy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, 4);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
        int cb, ob, ks;
        decode(p, item, cb, ob, ks);
        const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
        const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
        int tw = tile0 % p.tiles_w, t2 = tile0 / p.tiles_w;
        int th = t2 % p.tiles_h, n = t2 / p.tiles_h;
        for (int tile = tile0; tile < tile1; ++tile) {
          ptx::mbar_wait(&empty[s], ph ^ 1);
          ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)stage_bytes);
          uint8_t* dst = smem + s * stage_bytes;
          ptx::tma_load_4d(dst, &tmX, &full[s], cb * 64, tw * TILE_W - 1, th * TILE_H - 1, n);
          ptx::tma_load_4d(dst + X_BYTES, &tmDy, &full[s], ob * 64, tw * TILE_W, th * TILE_H, n);
          if (++s == p.stages) { s = 0; ph ^= 1; }
          if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++n; } }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    const uint32_t idesc128 = ptx::make_idesc_bf16(128, 64, 1, 1);
    const uint32_t idesc64 = ptx::make_idesc_bf16(64, 64, 1, 1);
    constexpr uint32_t nb_cols = 64;
    constexpr uint32_t dy_lbo = (1024u >> 4) << 16;              // unused for N = 64 (one 64-channel block)
    const uint32_t full_s = ptx::smem_u32(full), empty_s = ptx::smem_u32(empty);
    const uint32_t hi = ptx::desc_hi(1024);
    const uint32_t base_lo = (ptx::smem_u32(smem) & 0x3FFFFu) >> 4;
    constexpr uint32_t LBO_DX = (128u >> 4) << 16;               // pair (dx, dx+1): 128 B apart
    constexpr uint32_t LBO_DY = ((HALO_W * 128u) >> 4) << 16;    // pair (dy, dy+1): one halo row apart
    constexpr uint32_t ROW = (HALO_W * 128) >> 4;                // halo row pitch in 16-byte units
    int s = 0, it = 0;
    uint32_t ph = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int cb, ob, ks;
      decode(p, item, cb, ob, ks);
      const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
      const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
      ptx::mbar_wait(tempty, (it & 1) ^ 1);
      ptx::tc_fence_after();
      uint32_t accumulate = 0;
      for (int tile = tile0; tile < tile1; ++tile) {
        ptx::mbar_wait_s(full_s + s * 8, ph);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t x_lo = base_lo + s * ((uint32_t)stage_bytes >> 4);
          const uint32_t y_lo = x_lo + (X_BYTES >> 4);
#pragma unroll
          for (int kk = 0; kk < TILE_H; ++kk) {      // K step = one tile row of 16 pixels
            const uint32_t acc = kk ? 1u : accumulate;
            const uint32_t b = y_lo + kk * ((TILE_W * 128) >> 4);
            const uint64_t db = ptx::pack_desc(b | dy_lbo, hi);
            const uint32_t xr = x_lo + kk * ROW;     // halo pixel (kk, 0): tap (dy,dx) starts at (kk+dy, dx)
            // accumulators: 0 = taps (0,1), 1 = taps (3,4), 2 = taps (6,7), 3 = taps (2,5), 4 = tap 8
            ptx::umma_bf16(tmem_base + 0 * nb_cols, ptx::pack_desc((xr + 0 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
            ptx::umma_bf16(tmem_base + 1 * nb_cols, ptx::pack_desc((xr + 1 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
            ptx::umma_bf16(tmem_base + 2 * nb_cols, ptx::pack_desc((xr + 2 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
            ptx::umma_bf16(tmem_base + 3 * nb_cols, ptx::pack_desc((xr + 0 * ROW + 2 * 8) | LBO_DY, hi), db, idesc128, acc);
            ptx::umma_bf16(tmem_base + 4 * 64, ptx::pack_desc((xr + 2 * ROW + 2 * 8) | LBO_DX, hi), db, idesc64, acc);
          }
          ptx::umma_commit_s(empty_s + s * 8);
        }
        accumulate = 1;
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
      if (ptx::elect_one()) ptx::umma_commit(tfull);
      __syncwarp();
    }
  } else {
    // ============================== epilogue (warps 2..5) ==============================
    const int lg = warp & 3;
    int it = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int cb, ob, ks;
      decode(p, item, cb, ob, ks);
      ptx::mbar_wait(tfull, it & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
      for (int a = 0; a < NACC; ++a) {
        // which (tap, cin) does this thread's TMEM lane hold?
        int tap, cl;
        bool ok = true;
        if (a < 4) {                       // M = 128: lane group 0,1 -> first tap, 2,3 -> second tap
          const int first = a < 3 ? 3 * a : 2, second = a < 3 ? 3 * a + 1 : 5;
          tap = lg < 2 ? first : second;
          cl = (lg & 1) * 32 + lane;
        } else {                           // M = 64: rows 16*lg + lane live in lanes 0..15 of lane group lg
          tap = 8;
          cl = lg * 16 + lane;
          ok = lane < 16;
        }
        const int cin = cb * 64 + cl;
        ok = ok && cin < p.Cin;
        for (int c0 = 0; c0 < 64; c0 += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32(t_addr + (uint32_t)(a * 64 + c0), r);
          ptx::tmem_ld_wait();
          if (ok) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const int cout = ob * 64 + c0 + e;
              if (cout < p.Cout) p.partial[(((long)ks * p.Cout + cout) * 9 + tap) * p.Cin + cin] = __uint_as_float(r[e]);
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
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}


// ------------------------------------------------------------------------------------------------------------------
// Second form: dy = M side (128 output channels), x halo = N side (3 taps x 32 input channels), see the file comment.
// ------------------------------------------------------------------------------------------------------------------
constexpr int X2_BYTES = HALO_W * HALO_H * 64;     // 15360: 32 channels per halo pixel, SWIZZLE_64B
constexpr int DY2_BYTES = 2 * DY_BYTES;            // 32768: two 64-channel boxes
constexpr int STAGE2_BYTES = X2_BYTES + DY2_BYTES; // 48128 = 47 * 1024
constexpr int N2 = 96;                             // 3 taps x 32 input channels per MMA

__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_halo2_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                   const __grid_constant__ HWParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.stages * STAGE2_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + MAX_STAGES;
  uint64_t* tfull = bars + 2 * MAX_STAGES;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmX);
    ptx::prefetch_tmap(&tmDy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, 4);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
        int cb, ob, ks;
        decode(p, item, cb, ob, ks);
        const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
        const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
        int tw = tile0 % p.tiles_w, t2 = tile0 / p.tiles_w;
        int th = t2 % p.tiles_h, n = t2 / p.tiles_h;
        for (int tile = tile0; tile < tile1; ++tile) {
          ptx::mbar_wait(&empty[s], ph ^ 1);
          ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)STAGE2_BYTES);
          uint8_t* dst = smem + s * STAGE2_BYTES;
          ptx::tma_load_4d(dst, &tmX, &full[s], cb * 32, tw * TILE_W - 1, th * TILE_H - 1, n);
          ptx::tma_load_4d(dst + X2_BYTES, &tmDy, &full[s], ob * 128, tw * TILE_W, th * TILE_H, n);
          ptx::tma_load_4d(dst + X2_BYTES + DY_BYTES, &tmDy, &full[s], ob * 128 + 64, tw * TILE_W, th * TILE_H, n);
          if (++s == p.stages) { s = 0; ph ^= 1; }
          if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++n; } }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    const uint32_t idesc = ptx::make_idesc_bf16(128, N2, 1, 1);
    const uint32_t full_s = ptx::smem_u32(full), empty_s = ptx::smem_u32(empty);
    const uint32_t hi_a = ptx::desc_hi(1024);                     // dy: SWIZZLE_128B, 8 pixels x 128 B per K-atom
    const uint32_t hi_b = ptx::desc_hi_sw64(512);                 // x : SWIZZLE_64B,  8 pixels x  64 B per K-atom
    const uint32_t base_lo = (ptx::smem_u32(smem) & 0x3FFFFu) >> 4;
    constexpr uint32_t LBO_A = ((uint32_t)DY_BYTES >> 4) << 16;   // second 64-channel dy box
    constexpr uint32_t LBO_B = (64u >> 4) << 16;                  // next tap of the kernel row = next halo pixel = 64 B
    constexpr uint32_t ROW2 = (HALO_W * 64) >> 4;                 // halo row pitch in 16-byte units
    int s = 0, it = 0;
    uint32_t ph = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int cb, ob, ks;
      decode(p, item, cb, ob, ks);
      const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
      const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
      ptx::mbar_wait(tempty, (it & 1) ^ 1);
      ptx::tc_fence_after();
      uint32_t accumulate = 0;
      for (int tile = tile0; tile < tile1; ++tile) {
        ptx::mbar_wait_s(full_s + s * 8, ph);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t x_lo = base_lo + s * ((uint32_t)STAGE2_BYTES >> 4);
          const uint32_t y_lo = x_lo + (X2_BYTES >> 4);
#pragma unroll
          for (int kk = 0; kk < TILE_H; ++kk) {      // K step = one tile row of 16 pixels
            const uint32_t acc = kk ? 1u : accumulate;
            const uint64_t da = ptx::pack_desc((y_lo + kk * ((TILE_W * 128) >> 4)) | LBO_A, hi_a);
            const uint32_t xr = x_lo + kk * ROW2;    // halo pixel (kk, 0): kernel row dy starts at halo row kk + dy
            ptx::umma_bf16(tmem_base + 0 * N2, da, ptx::pack_desc((xr + 0 * ROW2) | LBO_B, hi_b), idesc, acc);
            ptx::umma_bf16(tmem_base + 1 * N2, da, ptx::pack_desc((xr + 1 * ROW2) | LBO_B, hi_b), idesc, acc);
            ptx::umma_bf16(tmem_base + 2 * N2, da, ptx::pack_desc((xr + 2 * ROW2) | LBO_B, hi_b), idesc, acc);
          }
          ptx::umma_commit_s(empty_s + s * 8);
        }
        accumulate = 1;
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
      if (ptx::elect_one()) ptx::umma_commit(tfull);
      __syncwarp();
    }
  } else {
    // ============================== epilogue (warps 2..5) ==============================
    const int lg = warp & 3;                     // TMEM lanes 32*lg .. 32*lg+31 = output channels of the block
    int it = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
      int cb, ob, ks;
      decode(p, item, cb, ob, ks);
      ptx::mbar_wait(tfull, it & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
      const int cout = ob * 128 + lg * 32 + lane;
      float* dst = p.partial + (((long)ks * p.Cout + cout) * 9) * p.Cin + cb * 32;
#pragma unroll 1
      for (int tap = 0; tap < 9; ++tap) {        // column (tap / 3) * 96 + (tap % 3) * 32 + ci  ==  tap * 32 + ci
        uint32_t r[32];
        ptx::tmem_ld_32x32(t_addr + (uint32_t)(tap * 32), r);
        ptx::tmem_ld_wait();
        if (cout < p.Cout) {
          float4* d4 = reinterpret_cast<float4*>(dst + (long)tap * p.Cin);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            d4[q] = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                                __uint_as_float(r[4 * q + 3]));
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}


// ------------------------------------------------------------------------------------------------------------------
// Third form: the second form on a CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2), for Cout % 256 == 0.
// One MMA is M = 256 (each CTA's 128 output channels from its own dy tile) x N = 96, and the B operand is SPLIT between
// the two CTAs: each CTA loads the x halo for 16 of the pair's 32 input channels (SWIZZLE_32B, 32-byte pixel pitch; the
// three taps of a kernel row are three 16-channel MN-atoms 32 bytes apart) and supplies 48 of the 96 columns -- per MMA a
// CTA reads 4 KB (A) + 1.5 KB (B half) from shared memory per 48 tensor-pipe cycles = 115 B/clk (second form: 146), and
// 40 KB instead of 47 KB from L2 per stage.  Only the leader CTA (cluster rank 0) issues MMAs; both CTAs run a TMA
// producer whose bytes are counted on the leader's full barrier, the leader's commit frees the stage in both CTAs
// (multicast arrive), both CTAs drain their own 128 TMEM lanes and arrive on the leader's TMEM-empty barrier.
// Accumulator columns of kernel row dy: dy*96 + n, n = half*48 + dx*16 + c  <->  tap (dy, dx), input channel half*16 + c.
// ------------------------------------------------------------------------------------------------------------------
constexpr int XP_BYTES = HALO_W * HALO_H * 32;         // 7680: 16 channels per halo pixel, SWIZZLE_32B
constexpr int STAGEP_BYTES = 40 * 1024;                // dy (32768, first: 1024-aligned) + x (7680) padded to 40 KB
constexpr int STAGEP_TX = DY2_BYTES + XP_BYTES;        // bytes ONE CTA's loads deliver per stage
constexpr int PAIR_STAGES = 5;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
wgrad_pair_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                  const __grid_constant__ HWParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PAIR_STAGES * STAGEP_BYTES);
  uint64_t* full = bars;                      // [PAIR_STAGES]  used in the leader only
  uint64_t* empty = bars + 8;                 // [PAIR_STAGES]  one per CTA, arrived by the leader's multicast commit
  uint64_t* tfull = bars + 16;                // one per CTA (multicast commit)
  uint64_t* tempty = bars + 17;               // leader's: 8 arrivals (4 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmX);
    ptx::prefetch_tmap(&tmDy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < PAIR_STAGES; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, 8);
    ptx::fence_barrier_init();
  }
  ptx::cluster_sync_all();                    // both CTAs' barriers exist before anything arrives on them remotely
  if (warp == 2) {
    ptx::tmem_alloc_pair(tmem_slot, 512);
    ptx::tmem_relinquish_pair();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer (both CTAs) ==============================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = pair; item < p.items; item += npairs) {
        int cb, ob, ks;
        decode(p, item, cb, ob, ks);
        const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
        const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
        int tw = tile0 % p.tiles_w, t2 = tile0 / p.tiles_w;
        int th = t2 % p.tiles_h, n = t2 / p.tiles_h;
        for (int tile = tile0; tile < tile1; ++tile) {
          ptx::mbar_wait_cluster(&empty[s], ph ^ 1);
          if (rank == 0) ptx::mbar_arrive_expect_tx(&full[s], 2u * STAGEP_TX);     // both CTAs' bytes land on this barrier
          uint8_t* dst = smem + s * STAGEP_BYTES;
          const int co = ob * 256 + (int)rank * 128;
          ptx::tma_load_4d_pair(dst, &tmDy, &full[s], co, tw * TILE_W, th * TILE_H, n);
          ptx::tma_load_4d_pair(dst + DY_BYTES, &tmDy, &full[s], co + 64, tw * TILE_W, th * TILE_H, n);
          ptx::tma_load_4d_pair(dst + DY2_BYTES, &tmX, &full[s], cb * 32 + (int)rank * 16, tw * TILE_W - 1, th * TILE_H - 1, n);
          if (++s == PAIR_STAGES) { s = 0; ph ^= 1; }
          if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++n; } }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer (leader CTA only) ==============================
    if (rank == 0) {
      const uint32_t idesc = ptx::make_idesc_bf16(256, N2, 1, 1);
      const uint32_t full_s = ptx::smem_u32(full), empty_s = ptx::smem_u32(empty);
      const uint32_t hi_a = ptx::desc_hi(1024);                    // dy: SWIZZLE_128B
      const uint32_t hi_b = ptx::desc_hi_sw32(256);                // x : SWIZZLE_32B, 8 pixels x 32 B per K-atom
      const uint32_t base_lo = (ptx::smem_u32(smem) & 0x3FFFFu) >> 4;
      constexpr uint32_t LBO_A = ((uint32_t)DY_BYTES >> 4) << 16;  // second 64-channel dy box
      constexpr uint32_t LBO_B = (32u >> 4) << 16;                 // next tap of the kernel row = next halo pixel = 32 B
      constexpr uint32_t ROWP = (HALO_W * 32) >> 4;                // halo row pitch in 16-byte units
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int item = pair; item < p.items; item += npairs, ++it) {
        int cb, ob, ks;
        decode(p, item, cb, ob, ks);
        const int tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
        const int tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
        ptx::mbar_wait_cluster(tempty, (it & 1) ^ 1);
        ptx::tc_fence_after();
        uint32_t accumulate = 0;
        for (int tile = tile0; tile < tile1; ++tile) {
          ptx::mbar_wait_cluster(&full[s], ph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t y_lo = base_lo + s * ((uint32_t)STAGEP_BYTES >> 4);
            const uint32_t x_lo = y_lo + (DY2_BYTES >> 4);
#pragma unroll
            for (int kk = 0; kk < TILE_H; ++kk) {
              const uint32_t acc = kk ? 1u : accumulate;
              const uint64_t da = ptx::pack_desc((y_lo + kk * ((TILE_W * 128) >> 4)) | LBO_A, hi_a);
              const uint32_t xr = x_lo + kk * ROWP;
              ptx::umma_bf16_pair(tmem_base + 0 * N2, da, ptx::pack_desc((xr + 0 * ROWP) | LBO_B, hi_b), idesc, acc);
              ptx::umma_bf16_pair(tmem_base + 1 * N2, da, ptx::pack_desc((xr + 1 * ROWP) | LBO_B, hi_b), idesc, acc);
              ptx::umma_bf16_pair(tmem_base + 2 * N2, da, ptx::pack_desc((xr + 2 * ROWP) | LBO_B, hi_b), idesc, acc);
            }
            ptx::umma_commit_pair(empty_s + s * 8, 3);             // frees stage s in BOTH CTAs
          }
          accumulate = 1;
          __syncwarp();
          if (++s == PAIR_STAGES) { s = 0; ph ^= 1; }
        }
        if (ptx::elect_one()) ptx::umma_commit_pair(ptx::smem_u32(tfull), 3);
        __syncwarp();
      }
    }
  } else {
    // ============================== epilogue (warps 2..5, both CTAs) ==============================
    const int lg = warp & 3;
    int it = 0;
    for (int item = pair; item < p.items; item += npairs, ++it) {
      int cb, ob, ks;
      decode(p, item, cb, ob, ks);
      ptx::mbar_wait_cluster(tfull, it & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16);
      const int cout = ob * 256 + (int)rank * 128 + lg * 32 + lane;
      float* dst = p.partial + (((long)ks * p.Cout + cout) * 9) * p.Cin + cb * 32;
#pragma unroll 1
      for (int j = 0; j < 9; ++j) {              // 32-column chunk j of the 288 accumulator columns
        uint32_t r[32];
        ptx::tmem_ld_32x32(t_addr + (uint32_t)(j * 32), r);
        ptx::tmem_ld_wait();
        if (cout < p.Cout) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {          // 16-column run: column c16 = 2*j + h of 18 runs
            const int run = 2 * j + h;
            const int dyk = run / 6, rr = run - dyk * 6;          // kernel row, run within the row's 96 columns
            const int half = rr / 3, dxk = rr - half * 3;         // which CTA's channels, tap within the row
            float4* d4 = reinterpret_cast<float4*>(dst + (long)(dyk * 3 + dxk) * p.Cin + half * 16);
#pragma unroll
            for (int q = 0; q < 4; ++q)
              d4[q] = make_float4(__uint_as_float(r[h * 16 + 4 * q]), __uint_as_float(r[h * 16 + 4 * q + 1]),
                                  __uint_as_float(r[h * 16 + 4 * q + 2]), __uint_as_float(r[h * 16 + 4 * q + 3]));
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(tempty, 0);          // the LEADER's barrier
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();                       // neither CTA may leave (or free TMEM) while its peer still uses the pair
  if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, 512);
}

void plan(const rbu_wgrad_args* a, HWParams* p) {
  memset(p, 0, sizeof(*p));
  p->N = a->N; p->H = a->H; p->W = a->W;
  p->tiles_w = rbu_cdiv(a->W, TILE_W);
  p->tiles_h = rbu_cdiv(a->H, TILE_H);
  p->tiles_total = p->tiles_w * p->tiles_h * a->N;
  p->Cout = a->Ca;
  p->Cin = a->Cb;
  {
    // Block shape: 128 output x 32 input channels (second form, balanced shared-memory operand fetch) whenever the channel
    // counts allow it, else 64 x 64 (the 64-output-channel level).
    const bool form2 = a->Ca % 128 == 0 && a->Cb % 32 == 0;
    p->OB = form2 ? 128 : 64;
    p->CB = form2 ? 32 : 64;
    if (form2 && a->Ca % 256 == 0) p->OB = 256;          // third form: a CTA pair per item
  }
  p->cin_blocks = rbu_cdiv(a->Cb, p->CB);
  p->cout_blocks = rbu_cdiv(a->Ca, p->OB);
  const int base_items = p->cin_blocks * p->cout_blocks;
  // Split-K factor from a cost model instead of a utilisation threshold (ncu on the first build of the second form:
  // 256 items on 148 SMs = 86.5 % of the SM-time busy, tensor pipe 72 % while busy but 59 % of the launch).  Every CTA
  // walks ceil(items / SMs) items of tiles_total / k tiles each; an item ends with an un-overlapped epilogue (147 KB of
  // partial sums) and every extra split adds one partial tensor for the ordered reduction kernel to read back.
  const int sms = p->OB == 256 ? rbu_num_sms() / 2 : rbu_num_sms();      // work items run on CTAs or on CTA pairs
  const double t_tile = p->OB == 128 ? 1550.0 : (p->OB == 256 ? 1400.0 : 1900.0);       // cycles per 8x16-pixel tile at the measured MMA efficiency
  const double t_epi = 6000.0;                                // TMEM -> global drain of one item
  const double out_bytes = (double)a->Ca * 9.0 * a->Cb * 4.0;
  const double t_red = out_bytes / (3.0e12 / 1.8e9);          // cycles per split: one more partial tensor for the reduction kernel
  int ks = 1;
  double best = 1e300;
  for (int k = 1; k <= p->tiles_total && (long)k * base_items <= 16L * sms; ++k) {
    const long items = (long)k * base_items;
    const long waves = (items + sms - 1) / sms;
    const double tiles_per_item = (double)p->tiles_total / k;
    if (k > 1 && tiles_per_item < 8.0) break;                 // items shorter than the 4-stage pipeline fill
    const double cost = (double)waves * (tiles_per_item * t_tile + t_epi) + (double)k * t_red;
    if (cost < best * (1.0 - 1e-9)) { best = cost; ks = k; }
  }
  p->ksplit = ks;
  p->items = base_items * ks;
}

}  // namespace

int rbu_wgrad_halo_supported(const rbu_wgrad_args* a) {
  return a->taps == 9 && a->dil == 1 && !a->gather && a->H >= TILE_H && a->W >= TILE_W;
}

size_t rbu_wgrad_halo_workspace_bytes(const rbu_wgrad_args* a) {
  HWParams p;
  plan(a, &p);
  size_t own = (size_t)p.ksplit * a->Ca * 9 * a->Cb * sizeof(float);
  return (own + 255) & ~(size_t)255;
}

// Argument validation is done by the caller (rbu_wgrad_gemm).
int rbu_wgrad_halo_launch(const rbu_wgrad_args* a, void* workspace, cudaStream_t stream) {
  HWParams p;
  plan(a, &p);
  p.partial = reinterpret_cast<float*>(workspace);
  const bool form2 = p.OB == 128, pairf = p.OB == 256;
  CUtensorMap tmX, tmDy;
  {
    const uint64_t dims[4] = {(uint64_t)a->Cb, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->b_ld * 2, (uint64_t)a->b_ld * 2 * a->W, (uint64_t)a->b_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {pairf ? 16u : (uint32_t)p.CB, HALO_W, HALO_H, 1};
    int rc = rbu_encode_tmap_bf16_sw(&tmX, a->b, 4, dims, str, box, pairf ? 32 : (form2 ? 64 : 128));
    if (rc) return rc;
  }
  {
    const uint64_t dims[4] = {(uint64_t)a->Ca, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->a_ld * 2, (uint64_t)a->a_ld * 2 * a->W, (uint64_t)a->a_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {64, TILE_W, TILE_H, 1};
    int rc = rbu_encode_tmap_bf16(&tmDy, a->a, 4, dims, str, box);
    if (rc) return rc;
  }
  const int stage_bytes = form2 ? STAGE2_BYTES : STAGE_BYTES;
  p.stages = MAX_STAGES;
  if (p.stages * stage_bytes + 1024 + 256 > SMEM_LIMIT) p.stages = (SMEM_LIMIT - 1024 - 256) / stage_bytes;
  const int smem_bytes = p.stages * stage_bytes + 1024 + 256;
  static std::atomic<unsigned long long> attr_set{0};      // one bit per device ordinal
  if (rbu_first_use_on_device(&attr_set)) {
    RBU_CHECK_CUDA(cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    RBU_CHECK_CUDA(cudaFuncSetAttribute(wgrad_halo2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  }
  if (pairf) {
    static std::atomic<unsigned long long> attr_pair{0};
    if (rbu_first_use_on_device(&attr_pair))
      RBU_CHECK_CUDA(cudaFuncSetAttribute(wgrad_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    const int pairs = rbu_num_sms() / 2;
    const int gridp = 2 * (p.items < pairs ? p.items : pairs);
    p.stages = PAIR_STAGES;
    wgrad_pair_kernel<<<gridp, NUM_THREADS, PAIR_STAGES * STAGEP_BYTES + 1024 + 256, stream>>>(tmX, tmDy, p);
    RBU_CHECK_LAUNCH();
    rbu_wgrad_reduce_launch(p.partial, p.ksplit, a->Ca, 9, a->Cb, a->out, a->accumulate, stream);
    RBU_CHECK_LAUNCH();
    return RBU_OK;
  }
  const int grid = p.items < rbu_num_sms() ? p.items : rbu_num_sms();
  if (form2)
    wgrad_halo2_kernel<<<grid, NUM_THREADS, smem_bytes, stream>>>(tmX, tmDy, p);
  else
    wgrad_halo_kernel<<<grid, NUM_THREADS, smem_bytes, stream>>>(tmX, tmDy, p);
  RBU_CHECK_LAUNCH();
  rbu_wgrad_reduce_launch(p.partial, p.ksplit, a->Ca, 9, a->Cb, a->out, a->accumulate, stream);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
