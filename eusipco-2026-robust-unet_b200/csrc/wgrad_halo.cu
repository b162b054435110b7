// K11, halo variant: weight gradient of a 3x3 (dilation 1) convolution on tcgen05 tensor cores with ALL NINE TAPS
// accumulated from ONE activation tile.
//
//   dW[cout][cin][tap] = sum over pixels p of  dy[p, cout] * x[p (+) tap, cin]
//
// The generic kernel (wgrad_gemm.cu) streams one shifted x tile per tap and, for 64-channel layers, runs M = 64 MMAs
// (half rate): 280-460 TFLOP/s on the 64-channel level, 750-850 elsewhere (L2->SM traffic bound, 98 FLOP/B).
// Here a work item is (a block of input channels) x (a block of output channels) x (a range of 8x16-pixel tiles), the x
// operand of a tile is its 10 x 24-slot halo (18 slots used), loaded by ONE TMA box and reused by all 9 taps through the
// start address of the MN-major UMMA descriptor (same trick as conv_halo.cu).  Split-K over tile ranges with fp32
// partials and the ordered reduction of wgrad_gemm.cu (deterministic).
// Replaces aten::convolution_backward(weight) of Main_Final.py:157,159,205-206.
//
// Structure: one persistent, warp-specialised body (wgrad_body<Form>, 192 threads, 1 CTA per SM) behind three entry
// points, one per form.  Warp 0 lane 0 is the TMA producer, warp 1 the MMA issuer, warps 2..5 drain the accumulators into
// the partials.  The forms share the work-item schedule, the shared-memory stage ring and the accumulator full / empty
// handoff; each supplies its stage layout (form_shape), its loads of one stage (load_stage), its MMAs for one 16-pixel
// tile row (mma_row) and its drain of one work item (drain).
//
// First form (wgrad_halo_kernel, Form::HALO, the 64-output-channel level): 64 input x 64 output channels per item.
//   * the x halo has 64 channels per pixel (3072-byte row pitch) and is the MMA's M side; two taps are stacked into one
//     M = 128 instruction: the descriptor's leading-byte-offset (distance between the two 64-channel column blocks) is
//     simply the distance between the two taps' start addresses in the halo buffer -- 128 B for (dx, dx+1), 3072 B for
//     (dy, dy+1).  Pairs (0,1) (3,4) (6,7) (2,5) and the single tap 8 (M = 64) give 5 accumulators x 64 columns = 320
//     TMEM columns;
//   * the dy operand (N = 64) is one plain 8x16-pixel box.
//   Per tile: 46 KB from L2 for 9.4 MFLOP (205 FLOP/B), 40 MMAs per barrier round trip.
//
// Second form (wgrad_halo2_kernel, Form::HALO2, used whenever Cout is a multiple of 128): the roles of the operands are
// swapped.  The first form runs M = 128 x N = 64 MMAs, which read 6 KB of operands from shared memory per 32 tensor-pipe
// cycles (192 B/clk against the 128 B/clk the SM delivers: ncu l1tex__data_pipe_tc_wavefronts_mem_shared 81 %, tensor
// pipe 50-61 %), and the 9 x 64 = 576 fp32 columns of a 64 x 64 x 9 block rule out N = 128 in the 512-column TMEM.  With
//   * dy as the M side (128 output channels = two 64-channel boxes, leading-byte-offset = one box) and
//   * the x halo as the N side, loaded with 32 channels per pixel (SWIZZLE_64B, 64-byte pixel pitch) so that the THREE
//     taps of a kernel row are three 32-channel MN-atoms 64 bytes apart: N = 96 with leading-byte-offset = 64 B,
// a work item is 128 output channels x 32 input channels x 9 taps = 3 accumulators x 96 columns (288 of 512), every MMA
// is M128 x N96 x K16 (7 KB per 48 cycles = 146 B/clk) and the L2 traffic per FLOP is unchanged (47 KB per 9.4 MFLOP).
// The epilogue thread (= output channel) reads, per tap, 32 consecutive input channels = one 128-byte run of the partials.
//
// Third form (wgrad_pair_kernel, Form::PAIR): the second form on a CTA PAIR (thread-block cluster of 2, tcgen05
// cta_group::2), for Cout % 256 == 0.  One MMA is M = 256 (each CTA's 128 output channels from its own dy tile) x N = 96,
// and the B operand is SPLIT between the two CTAs: each CTA loads the x halo for 16 of the pair's 32 input channels
// (SWIZZLE_32B, 32-byte pixel pitch; the three taps of a kernel row are three 16-channel MN-atoms 32 bytes apart) and
// supplies 48 of the 96 columns -- per MMA a CTA reads 4 KB (A) + 1.5 KB (B half) from shared memory per 48 tensor-pipe
// cycles = 115 B/clk (second form: 146), and 40 KB instead of 47 KB from L2 per stage.  Only the leader CTA (cluster rank
// 0) issues MMAs; both CTAs run a TMA producer whose bytes are counted on the leader's full barrier, the leader's commit
// frees the stage in both CTAs (multicast arrive), both CTAs drain their own 128 TMEM lanes and arrive on the leader's
// TMEM-empty barrier.  Every barrier wait of this form is a cluster-scope acquire.
// Accumulator columns of kernel row dy: dy*96 + n, n = half*48 + dx*16 + c  <->  tap (dy, dx), input channel half*16 + c.
#include "rbu_common.cuh"
#include "rbu_ptx.cuh"
#include "tma_host.cuh"

namespace {

constexpr int TILE_W = 16, TILE_H = 8;
constexpr int HALO_W = 24, HALO_H = 10;
constexpr int DY_BYTES = TILE_W * TILE_H * 128;        // 16384: one 64-channel dy box
constexpr int DY2_BYTES = 2 * DY_BYTES;                // 32768: two 64-channel boxes
constexpr int X_BYTES = HALO_W * HALO_H * 128;         // 30720: first form, 64 channels per halo pixel, SWIZZLE_128B
constexpr int X2_BYTES = HALO_W * HALO_H * 64;         // 15360: second form, 32 channels per halo pixel, SWIZZLE_64B
constexpr int XP_BYTES = HALO_W * HALO_H * 32;         // 7680: pair form, 16 channels per halo pixel, SWIZZLE_32B
constexpr int NUM_THREADS = 192;
constexpr int SMEM_LIMIT = 232448;
constexpr int SMEM_RESERVE = 1024 + 256;               // alignment of the ring + barriers and the TMEM address slot
constexpr int N2 = 96;                                 // second and pair form: 3 taps x 32 input channels per MMA

enum class Form : int { HALO, HALO2, PAIR };

// Everything the host plan and the device body need to know about a form's shape.
struct FormShape {
  int CB, OB;          // input x output channels of a work item
  int xc;              // channels per pixel of one CTA's x halo box (its pixel pitch, 2 * xc bytes, is the swizzle span)
  int stage_bytes;     // stride of the shared-memory stage ring (multiple of 1024)
  int tx_bytes;        // bytes one stage's TMA loads deliver to the (leader's) full barrier
  int stages;          // ring depth
  double t_tile;       // split-K cost model: cycles per 8x16-pixel tile at the measured MMA efficiency
};

__host__ __device__ constexpr int ring_depth(int want, int stage_bytes) {
  return want * stage_bytes + SMEM_RESERVE <= SMEM_LIMIT ? want : (SMEM_LIMIT - SMEM_RESERVE) / stage_bytes;
}

__host__ __device__ constexpr FormShape form_shape(Form f) {
  // stage layouts: HALO = x halo | dy;  HALO2 = x halo | dy | dy;  PAIR = dy | dy | x halo, padded to 40 KB
  return f == Form::HALO    ? FormShape{64, 64, 64, X_BYTES + DY_BYTES, X_BYTES + DY_BYTES,
                                        ring_depth(4, X_BYTES + DY_BYTES), 1900.0}
         : f == Form::HALO2 ? FormShape{32, 128, 32, X2_BYTES + DY2_BYTES, X2_BYTES + DY2_BYTES,
                                        ring_depth(4, X2_BYTES + DY2_BYTES), 1550.0}
                            : FormShape{32, 256, 16, 40 * 1024, 2 * (DY2_BYTES + XP_BYTES), ring_depth(5, 40 * 1024), 1400.0};
}

struct HWParams {
  int N, H, W;
  int tiles_w, tiles_h, tiles_total;
  int Cout, Cin;
  int cin_blocks, cout_blocks, ksplit, items;
  Form form;
  float* partial;   // [ksplit][Cout][9][Cin]
};

// The tile schedule: work item -> (input-channel block cb, output-channel block ob, split ks) -> tiles [tile0, tile1).
struct WorkItem {
  int cb, ob, ks, tile0, tile1;
  __device__ __forceinline__ WorkItem(const HWParams& p, int item) {
    cb = item % p.cin_blocks; item /= p.cin_blocks;
    ob = item % p.cout_blocks;
    ks = item / p.cout_blocks;
    tile0 = (int)((long)ks * p.tiles_total / p.ksplit);
    tile1 = (int)((long)(ks + 1) * p.tiles_total / p.ksplit);
  }
};

// Position (tw, th, n) of a tile, stepped through the tile range in order.
struct TileCursor {
  int tw, th, n;
  __device__ __forceinline__ TileCursor(const HWParams& p, int tile) {
    tw = tile % p.tiles_w;
    const int t2 = tile / p.tiles_w;
    th = t2 % p.tiles_h;
    n = t2 / p.tiles_h;
  }
  __device__ __forceinline__ void next(const HWParams& p) {
    if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++n; } }
  }
};

// TMA loads of one stage (the tile at `c`) into `dst`, completing on `bar`.
template <Form F>
__device__ __forceinline__ void load_stage(uint8_t* dst, const CUtensorMap& tmX, const CUtensorMap& tmDy, uint64_t* bar,
                                           const WorkItem& w, const TileCursor& c, int rank) {
  const int x0 = c.tw * TILE_W, y0 = c.th * TILE_H;
  if constexpr (F == Form::HALO) {
    ptx::load_4d<false>(dst, &tmX, bar, w.cb * 64, x0 - 1, y0 - 1, c.n);
    ptx::load_4d<false>(dst + X_BYTES, &tmDy, bar, w.ob * 64, x0, y0, c.n);
  } else if constexpr (F == Form::HALO2) {
    ptx::load_4d<false>(dst, &tmX, bar, w.cb * 32, x0 - 1, y0 - 1, c.n);
    ptx::load_4d<false>(dst + X2_BYTES, &tmDy, bar, w.ob * 128, x0, y0, c.n);
    ptx::load_4d<false>(dst + X2_BYTES + DY_BYTES, &tmDy, bar, w.ob * 128 + 64, x0, y0, c.n);
  } else {
    const int co = w.ob * 256 + rank * 128;
    ptx::load_4d<true>(dst, &tmDy, bar, co, x0, y0, c.n);
    ptx::load_4d<true>(dst + DY_BYTES, &tmDy, bar, co + 64, x0, y0, c.n);
    ptx::load_4d<true>(dst + DY2_BYTES, &tmX, bar, w.cb * 32 + rank * 16, x0 - 1, y0 - 1, c.n);
  }
}

// The MMAs of tile row kk (K step = one row of 16 pixels) on the stage at shared address st (16-byte units).
template <Form F>
__device__ __forceinline__ void mma_row(uint32_t tmem_base, uint32_t st, int kk, uint32_t acc) {
  constexpr uint32_t DY_ROW = (TILE_W * 128) >> 4;               // one 16-pixel row of a dy box
  if constexpr (F == Form::HALO) {
    constexpr uint32_t dy_lbo = (1024u >> 4) << 16;              // unused for N = 64 (one 64-channel block)
    constexpr uint32_t LBO_DX = (128u >> 4) << 16;               // pair (dx, dx+1): 128 B apart
    constexpr uint32_t LBO_DY = ((HALO_W * 128u) >> 4) << 16;    // pair (dy, dy+1): one halo row apart
    constexpr uint32_t ROW = (HALO_W * 128) >> 4;                // halo row pitch in 16-byte units
    const uint32_t idesc128 = ptx::make_idesc_bf16(128, 64, 1, 1);
    const uint32_t idesc64 = ptx::make_idesc_bf16(64, 64, 1, 1);
    const uint32_t hi = ptx::desc_hi(1024);
    const uint64_t db = ptx::pack_desc((st + (X_BYTES >> 4) + kk * DY_ROW) | dy_lbo, hi);
    const uint32_t xr = st + kk * ROW;                           // halo pixel (kk, 0): tap (dy,dx) starts at (kk+dy, dx)
    // accumulators: 0 = taps (0,1), 1 = taps (3,4), 2 = taps (6,7), 3 = taps (2,5), 4 = tap 8
    ptx::umma_bf16(tmem_base + 0 * 64, ptx::pack_desc((xr + 0 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
    ptx::umma_bf16(tmem_base + 1 * 64, ptx::pack_desc((xr + 1 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
    ptx::umma_bf16(tmem_base + 2 * 64, ptx::pack_desc((xr + 2 * ROW + 0 * 8) | LBO_DX, hi), db, idesc128, acc);
    ptx::umma_bf16(tmem_base + 3 * 64, ptx::pack_desc((xr + 0 * ROW + 2 * 8) | LBO_DY, hi), db, idesc128, acc);
    ptx::umma_bf16(tmem_base + 4 * 64, ptx::pack_desc((xr + 2 * ROW + 2 * 8) | LBO_DX, hi), db, idesc64, acc);
  } else {
    // dy is the M side (SWIZZLE_128B, second 64-channel box one box further), the x halo the N side: kernel row dy
    // starts at halo row kk + dy, and its three taps are consecutive halo pixels
    constexpr bool PAIR = F == Form::PAIR;
    constexpr uint32_t XPIX = 2 * form_shape(F).xc;               // halo pixel pitch in bytes
    constexpr uint32_t ROWX = (HALO_W * XPIX) >> 4;               // halo row pitch in 16-byte units
    constexpr uint32_t LBO_A = ((uint32_t)DY_BYTES >> 4) << 16;   // second 64-channel dy box
    constexpr uint32_t LBO_B = (XPIX >> 4) << 16;                 // next tap of the kernel row = next halo pixel
    const uint32_t idesc = ptx::make_idesc_bf16(PAIR ? 256 : 128, N2, 1, 1);
    const uint32_t hi_a = ptx::desc_hi(1024);
    const uint32_t hi_b = PAIR ? ptx::desc_hi_sw32(8 * XPIX) : ptx::desc_hi_sw64(8 * XPIX);   // 8 pixels per K-atom
    const uint32_t y_lo = PAIR ? st : st + (X2_BYTES >> 4);
    const uint32_t x_lo = PAIR ? st + (DY2_BYTES >> 4) : st;
    const uint64_t da = ptx::pack_desc((y_lo + kk * DY_ROW) | LBO_A, hi_a);
    const uint32_t xr = x_lo + kk * ROWX;
    ptx::mma<PAIR>(tmem_base + 0 * N2, da, ptx::pack_desc((xr + 0 * ROWX) | LBO_B, hi_b), idesc, acc);
    ptx::mma<PAIR>(tmem_base + 1 * N2, da, ptx::pack_desc((xr + 1 * ROWX) | LBO_B, hi_b), idesc, acc);
    ptx::mma<PAIR>(tmem_base + 2 * N2, da, ptx::pack_desc((xr + 2 * ROWX) | LBO_B, hi_b), idesc, acc);
  }
}

// Epilogue warp `lg` (TMEM lanes 32 lg .. 32 lg + 31 at t_addr) stores its part of work item w's accumulators.
template <Form F>
__device__ __forceinline__ void drain(const HWParams& p, uint32_t t_addr, int lg, int lane, int rank, const WorkItem& w) {
  if constexpr (F == Form::HALO) {
    for (int a = 0; a < 5; ++a) {
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
      const int cin = w.cb * 64 + cl;
      ok = ok && cin < p.Cin;
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r[32];
        ptx::tmem_ld_32x32(t_addr + (uint32_t)(a * 64 + c0), r);
        ptx::tmem_ld_wait();
        if (ok) {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int cout = w.ob * 64 + c0 + e;
            if (cout < p.Cout) p.partial[(((long)w.ks * p.Cout + cout) * 9 + tap) * p.Cin + cin] = __uint_as_float(r[e]);
          }
        }
      }
    }
  } else {
    // TMEM lane = output channel; each thread writes 32-column chunks as runs of consecutive input channels
    const int cout = w.ob * form_shape(F).OB + rank * 128 + lg * 32 + lane;
    float* dst = p.partial + (((long)w.ks * p.Cout + cout) * 9) * p.Cin + w.cb * 32;
#pragma unroll 1
    for (int j = 0; j < 9; ++j) {              // 32-column chunk j of the 288 accumulator columns
      uint32_t r[32];
      ptx::tmem_ld_32x32(t_addr + (uint32_t)(j * 32), r);
      ptx::tmem_ld_wait();
      if (cout < p.Cout) {
        if constexpr (F == Form::HALO2) {      // column (tap / 3) * 96 + (tap % 3) * 32 + ci  ==  tap * 32 + ci
          float4* d4 = reinterpret_cast<float4*>(dst + (long)j * p.Cin);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            d4[q] = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                                __uint_as_float(r[4 * q + 3]));
        } else {
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
    }
  }
}

template <Form F>
__device__ __forceinline__ void wgrad_body(const CUtensorMap& tmX, const CUtensorMap& tmDy, const HWParams& p) {
  constexpr bool PAIR = F == Form::PAIR;
  constexpr FormShape S = form_shape(F);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S.stages * S.stage_bytes);   // [stages]  PAIR: used in the leader only
  uint64_t* empty = full + S.stages;        // [stages]  PAIR: one per CTA, arrived by the leader's multicast commit
  uint64_t* tfull = empty + S.stages;       // PAIR: one per CTA (multicast commit)
  uint64_t* tempty = tfull + 1;             // PAIR: the leader's, 8 arrivals (4 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = PAIR ? (int)ptx::cluster_ctarank() : 0;
  const int first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // first work item and stride of this CTA (pair)
  const int step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmX);
    ptx::prefetch_tmap(&tmDy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S.stages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    ptx::mbar_init(tfull, 1);
    ptx::mbar_init(tempty, PAIR ? 8 : 4);
    ptx::fence_barrier_init();
  }
  if (PAIR) ptx::cluster_sync_all();        // both CTAs' barriers exist before anything arrives on them remotely
  if (warp == 2) {
    if (PAIR) {
      ptx::tmem_alloc_pair(tmem_slot, 512);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(tmem_slot, 512);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer (PAIR: both CTAs) ==============================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = first; item < p.items; item += step) {
        const WorkItem w(p, item);
        TileCursor c(p, w.tile0);
        for (int tile = w.tile0; tile < w.tile1; ++tile) {
          ptx::bar_wait_remote<PAIR>(&empty[s], ph ^ 1);
          if (rank == 0) ptx::mbar_arrive_expect_tx(&full[s], (uint32_t)S.tx_bytes);   // PAIR: both CTAs' bytes
          load_stage<F>(smem + s * S.stage_bytes, tmX, tmDy, &full[s], w, c, rank);
          if (++s == S.stages) { s = 0; ph ^= 1; }
          c.next(p);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer (PAIR: the leader CTA only) ==============================
    if (rank == 0) {
      const uint32_t full_s = ptx::smem_u32(full), empty_s = ptx::smem_u32(empty);
      const uint32_t base_lo = (ptx::smem_u32(smem) & 0x3FFFFu) >> 4;
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int item = first; item < p.items; item += step, ++it) {
        const WorkItem w(p, item);
        ptx::bar_wait_remote<PAIR>(tempty, (it & 1) ^ 1);
        ptx::tc_fence_after();
        uint32_t accumulate = 0;
        for (int tile = w.tile0; tile < w.tile1; ++tile) {
          if (PAIR) ptx::mbar_wait_cluster_s(full_s + s * 8, ph); else ptx::mbar_wait_s(full_s + s * 8, ph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t st = base_lo + s * ((uint32_t)S.stage_bytes >> 4);
#pragma unroll
            for (int kk = 0; kk < TILE_H; ++kk) mma_row<F>(tmem_base, st, kk, kk ? 1u : accumulate);
            ptx::commit_s<PAIR>(empty_s + s * 8);                  // PAIR: frees stage s in BOTH CTAs
          }
          accumulate = 1;
          __syncwarp();
          if (++s == S.stages) { s = 0; ph ^= 1; }
        }
        if (ptx::elect_one()) ptx::commit_s<PAIR>(ptx::smem_u32(tfull));
        __syncwarp();
      }
    }
  } else {
    // ============================== epilogue (warps 2..5; PAIR: both CTAs) ==============================
    const int lg = warp & 3;
    int it = 0;
    for (int item = first; item < p.items; item += step, ++it) {
      const WorkItem w(p, item);
      ptx::bar_wait_remote<PAIR>(tfull, it & 1);
      ptx::tc_fence_after();
      drain<F>(p, tmem_base + ((uint32_t)(lg * 32) << 16), lg, lane, rank, w);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) ptx::mbar_arrive_cluster(tempty, 0); else ptx::mbar_arrive(tempty);   // PAIR: the LEADER's barrier
      }
    }
  }
  ptx::tc_fence_before();
  if (PAIR) {
    ptx::cluster_sync_all();                // neither CTA may leave (or free TMEM) while its peer still uses the pair
    if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, 512);
  } else {
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
  }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_halo_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                  const __grid_constant__ HWParams p) {
  wgrad_body<Form::HALO>(tmX, tmDy, p);
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
wgrad_halo2_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                   const __grid_constant__ HWParams p) {
  wgrad_body<Form::HALO2>(tmX, tmDy, p);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
wgrad_pair_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDy,
                  const __grid_constant__ HWParams p) {
  wgrad_body<Form::PAIR>(tmX, tmDy, p);
}

void plan(const rbu_wgrad_args* a, HWParams* p) {
  memset(p, 0, sizeof(*p));
  p->N = a->N; p->H = a->H; p->W = a->W;
  p->tiles_w = rbu_cdiv(a->W, TILE_W);
  p->tiles_h = rbu_cdiv(a->H, TILE_H);
  p->tiles_total = p->tiles_w * p->tiles_h * a->N;
  p->Cout = a->Ca;
  p->Cin = a->Cb;
  // Form: 128 output x 32 input channels (second form, balanced shared-memory operand fetch) whenever the channel counts
  // allow it, on a CTA pair when Cout is also a multiple of 256, else 64 x 64 (the 64-output-channel level).
  if (a->Ca % 128 == 0 && a->Cb % 32 == 0)
    p->form = a->Ca % 256 == 0 ? Form::PAIR : Form::HALO2;
  else
    p->form = Form::HALO;
  const FormShape f = form_shape(p->form);
  p->cin_blocks = rbu_cdiv(a->Cb, f.CB);
  p->cout_blocks = rbu_cdiv(a->Ca, f.OB);
  const int base_items = p->cin_blocks * p->cout_blocks;
  // Split-K factor from a cost model instead of a utilisation threshold (ncu on the first build of the second form:
  // 256 items on 148 SMs = 86.5 % of the SM-time busy, tensor pipe 72 % while busy but 59 % of the launch).  Every CTA
  // walks ceil(items / SMs) items of tiles_total / k tiles each; an item ends with an un-overlapped epilogue (147 KB of
  // partial sums) and every extra split adds one partial tensor for the ordered reduction kernel to read back.
  const int sms = p->form == Form::PAIR ? rbu_num_sms() / 2 : rbu_num_sms();   // work items run on CTAs or on CTA pairs
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
    const double cost = (double)waves * (tiles_per_item * f.t_tile + t_epi) + (double)k * t_red;
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
  const FormShape f = form_shape(p.form);
  CUtensorMap tmX, tmDy;
  {
    const uint64_t dims[4] = {(uint64_t)a->Cb, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->b_ld * 2, (uint64_t)a->b_ld * 2 * a->W, (uint64_t)a->b_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {(uint32_t)f.xc, HALO_W, HALO_H, 1};
    int rc = rbu_encode_tmap_bf16_sw(&tmX, a->b, 4, dims, str, box, 2 * f.xc);
    if (rc) return rc;
  }
  {
    const uint64_t dims[4] = {(uint64_t)a->Ca, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->a_ld * 2, (uint64_t)a->a_ld * 2 * a->W, (uint64_t)a->a_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {64, TILE_W, TILE_H, 1};
    int rc = rbu_encode_tmap_bf16(&tmDy, a->a, 4, dims, str, box);
    if (rc) return rc;
  }
  void (*kernel)(CUtensorMap, CUtensorMap, HWParams) =
      p.form == Form::HALO ? wgrad_halo_kernel : p.form == Form::HALO2 ? wgrad_halo2_kernel : wgrad_pair_kernel;
  static std::atomic<unsigned long long> attr_set[3]{};     // per form: one bit per device ordinal
  if (rbu_first_use_on_device(&attr_set[(int)p.form]))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  const int cta_per_item = p.form == Form::PAIR ? 2 : 1;
  const int units = rbu_num_sms() / cta_per_item;           // CTAs or CTA pairs
  const int grid = cta_per_item * (p.items < units ? p.items : units);
  kernel<<<grid, NUM_THREADS, f.stages * f.stage_bytes + SMEM_RESERVE, stream>>>(tmX, tmDy, p);
  RBU_CHECK_LAUNCH();
  rbu_wgrad_reduce_launch(p.partial, p.ksplit, a->Ca, 9, a->Cb, a->out, a->accumulate, stream);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
