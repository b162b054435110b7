// K1 / K10, halo variant: 3x3 (dilation 1) and 1x1 convolutions and their data gradients as an implicit GEMM on
// tcgen05 tensor cores where every activation tile is fetched from L2 ONCE and reused by all nine taps, and every
// weight tile is used for TWO 128-pixel MMA tiles.
//
// The generic kernel (conv_gemm.cu) issues one TMA load of the 128-pixel x 64-channel A tile per tap, i.e. nine
// loads of (almost) the same pixels per 64-channel slab.  Here the output tile is 16 rows x 16 columns of one image
// and the A operand is its 18 x 24(18 used) x 64-channel halo, loaded by ONE 4-D TMA box into a SWIZZLE_128B buffer with
// a 3072-byte row pitch.  Tap (dy,dx) of the left / right 8-column half of the tile is then just a different START
// ADDRESS of the same buffer: the UMMA shared-memory descriptor (K-major, 8-pixel row groups, stride-byte-offset = 3072
// = one halo row) starts at pixel (dy, dx + 8*half) of the halo; the start is a multiple of 128 B, not of 1024 B.
// Measured on B200: the tensor core applies the 128-byte swizzle XOR from the ABSOLUTE shared-memory address bits
// [7:9] of every row it fetches -- exactly what TMA did when it wrote the rows -- so the descriptor's
// matrix-base-offset field stays 0 (setting it to (start >> 7) & 7 double-counts the phase: every 3x3 parity test
// failed with it, all pass without).
//
// Why 256 pixels per weight tile: with one 128-pixel tile per CTA the >= 128-channel layers re-read K x N x 2 bytes of
// weights from L2 per tile, and every such layer sat at 42 +- 1 bytes / clk / SM of L2 -> SM traffic (128->128: 1300,
// 256->256: 1500, 512->512: 1530 TFLOP/s; the chip-wide L2 ceiling of ~6300 B/clk), not at the tensor pipe.  Two
// accumulators per weight stage halve that traffic.
//
// Structure (persistent, warp specialised, 320 threads, 1 CTA / SM):
//   warp 0 lane 0 : TMA producer -- A ring (halo tiles, 2 stages) and B ring (weight tiles, 1 or 3 taps per stage)
//   warp 1        : MMA issuer   -- per slab 9 taps x 2 halves x 4 tcgen05.mma (K = 16); accumulators rotate through
//                                   512 / block_n TMEM slots (4 for block_n <= 128, 2 for 256)
//   warps 2..9    : epilogue     -- warps 2-5 drain the left half-tile, 6-9 the right one (tcgen05.ld, bias / addend /
//                                   ReLU, bf16 pack, 16-byte stores; gemm_epilogue.cuh)
// Two accumulated segments are supported (conv1 3x3 dgrad + shortcut 1x1 dgrad; 1x1 segments use a plain
// 16 x 16-pixel box with a 2048-byte pitch).
// Replaces aten::convolution / convolution_backward(input) of Main_Final.py:157,159,172,126,131.
#include "rbu_common.cuh"
#include "rbu_ptx.cuh"
#include "tma_host.cuh"
#include "gemm_epilogue.cuh"

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int TILE_W = 16, TILE_H = 16, HALF_W = 8;
#ifndef RBU_HALO_W
#define RBU_HALO_W 24
#endif
constexpr int HALO_W = RBU_HALO_W, HALO_H = 18;       // halo row pitch in pixel slots (18 used)
constexpr int A_HALO_TX = HALO_H * HALO_W * 128;      // bytes one halo box delivers
constexpr int A_HALO_BYTES = (A_HALO_TX + 1023) & ~1023;   // stage stride (1024-aligned swizzle phase)
constexpr int A_PLAIN_BYTES = TILE_H * TILE_W * 128;  // 32768
constexpr int NUM_THREADS = 320;   // TMA warp, MMA warp, 8 epilogue warps
constexpr int MAX_B_STAGES = 8;
constexpr int MAX_SLOTS = 4;
constexpr int STG_BYTES = 32 * 64 * 2;   // staging buffer of one epilogue warp: its 32 pixels x 64 channels (one TMA store box)
constexpr int SMEM_LIMIT = 232448 - EPI_STAT_FLOATS * 4;   // minus the static statistics accumulators
constexpr int LOOKAHEAD_TAP = 4;                      // the next slab's A tile is requested after this tap's B tile
constexpr uint32_t HALF_OFF = (HALF_W * 128) >> 4;    // right half-tile: 8 pixels = 1024 B further (descriptor units)
constexpr uint32_t ROW_OFF = (HALO_W * 128) >> 4;     // one halo row down

struct HParams {
  int N, H, W;
  int tiles_w, tiles_h;
  FastDiv fd_nb, fd_tw, fd_th;
  int n_blocks, block_n, Ncols;
  int slot_mask, slot_shift;   // TMEM accumulator slots: nslots = slot_mask + 1 = 1 << slot_shift
  int nseg;
  int taps[2], C[2];
  int a_stages, b_stages, tmem_cols, total_tiles;
  int sp_total;   // spatial tiles (tiles_w * tiles_h * N); a CTA pair's work unit is two of them times one column block
  int tps;   // taps per B stage for a 3x3 segment (3 = one kernel row per stage when block_n <= 128, else 1)
  int tma_store;  // 1: outputs leave through the y tensor map (8 x 4-pixel x 64-channel boxes staged in shared memory)
  int st_bufs;    // staging buffers per epilogue warp (1 or 2)
  int resident;   // 1: the whole weight operand (slabs x 9 taps) stays in shared memory for the life of the CTA
  bf16* y;
  long long y_ld;
  const float* bias;
  const float* scale;
  int relu;
  const bf16* addend;
  long long addend_ld;
  float* tile_stats;   // [N][tiles_h*tiles_w*2][4][Ncols]: per image and half-tile column sum / sum of squares / max / min
  float* stats;   // [SMs][2][Ncols] (one row per CTA) column sum / sum of squares of the stored output, or NULL
};

// Enumerates the (tile, segment, 64-channel slab) sequence of this CTA; producer and MMA issuer walk it in lockstep.
struct SlabIter {
  int tile, seg, kc, stride;
  bool valid;
  __device__ __forceinline__ void init(const HParams& p, int first, int step) {
    tile = first; seg = 0; kc = 0; stride = step;
    valid = tile < p.total_tiles;
  }
  __device__ __forceinline__ void next(const HParams& p) {
    if (++kc < (p.C[seg] + BLOCK_K - 1) / BLOCK_K) return;
    kc = 0;
    if (++seg < p.nseg) return;
    seg = 0;
    tile += stride;
    valid = tile < p.total_tiles;
  }
};

// PAIR: work unit `tile` = (two horizontally consecutive spatial tiles, one column block); CTA `rank` of the pair owns
// spatial tile 2 * (tile / n_blocks) + rank, which may lie past the end (odd tile count): the CTA still walks the
// schedule (its TMA boxes are out of bounds = zero fill) but stores nothing.
template <bool PAIR>
__device__ __forceinline__ bool tile_coords(const HParams& p, int tile, int rank, int& nb, int& w0, int& h0, int& n) {
  int sp = fast_div(tile, p.fd_nb);
  nb = tile - sp * p.n_blocks;
  if (PAIR) sp = 2 * sp + rank;
  const int q = fast_div(sp, p.fd_tw);
  w0 = (sp - q * p.tiles_w) * TILE_W;
  n = fast_div(q, p.fd_th);
  h0 = (q - n * p.tiles_h) * TILE_H;
  return !PAIR || sp < p.sp_total;
}

// PAIR = true: the kernel runs as thread-block clusters of two CTAs (cta_group::2).  Each CTA owns its own spatial tile
// (halo in its own shared memory = 128 + 128 of the M = 256 rows of every MMA) and HALF of the weight tile (block_n / 2
// output channels: the B operand of a pair MMA is split along N between the two CTAs' shared memory), so the weight
// bytes per SM -- L2 -> SM traffic and shared-memory operand fetch -- halve.  Only the leader (cluster rank 0) issues
// MMAs; its commits are multicast to both CTAs' empty / accumulator-full barriers, both CTAs' TMA loads count on the
// leader's full barriers, and both epilogues arrive on the leader's accumulator-empty barriers.
// Barriers completed by tcgen05.commit or TMA complete_tx are polled with the CTA-scope wait in both instantiations (the
// data they guard travels through the async proxy / TMEM); only the accumulator-empty barriers, which collect
// release.cluster arrivals from the peer CTA's epilogue threads, need the cluster-scope acquire (ptx::bar_wait_remote).
template <bool PAIR>
__device__ __forceinline__ void conv_halo_body(const CUtensorMap& tmA0, const CUtensorMap& tmB0, const CUtensorMap& tmA1,
                                               const CUtensorMap& tmB1, const CUtensorMap& tmY, const HParams& p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int rank = PAIR ? (int)ptx::cluster_ctarank() : 0;
  const int cta0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;        // first work unit and stride of this CTA (pair)
  const int cta_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int bn_cta = PAIR ? p.block_n >> 1 : p.block_n;   // weight rows (output channels) in this CTA's shared memory
  const int b_bytes = bn_cta * 128;             // one tap's weight tile
  const int bs_bytes = b_bytes * p.tps;         // one B stage
  uint8_t* smA = smem;
  uint8_t* smB = smem + p.a_stages * A_HALO_BYTES;
  uint8_t* stg_base = smB + p.b_stages * bs_bytes;                          // 1024-aligned: all regions are multiples of 2 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + (p.tma_store ? 8 * p.st_bufs * STG_BYTES : 0));
  uint64_t* fullA = bars;                      // [4]
  uint64_t* emptyA = bars + 4;                 // [4]
  uint64_t* fullB = bars + 8;                  // [MAX_B_STAGES]
  uint64_t* emptyB = bars + 8 + MAX_B_STAGES;  // [MAX_B_STAGES]
  uint64_t* tfull = bars + 8 + 2 * MAX_B_STAGES;   // [MAX_SLOTS]
  uint64_t* tempty = tfull + MAX_SLOTS;            // [MAX_SLOTS]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + MAX_SLOTS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  __shared__ __align__(16) float stat_smem[EPI_STAT_FLOATS];
  if (p.stats)
    for (int i = threadIdx.x; i < EPI_STAT_FLOATS; i += NUM_THREADS) stat_smem[i] = 0.f;
  static_assert(EPI_STAT_FLOATS >= 2 * 2 * 4 * 4 * 32, "tile statistics exchange buffer");

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA0);
    ptx::prefetch_tmap(&tmB0);
    if (p.tma_store) ptx::prefetch_tmap(&tmY);
    if (p.nseg > 1) {
      ptx::prefetch_tmap(&tmA1);
      ptx::prefetch_tmap(&tmB1);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.a_stages; ++s) {
      ptx::mbar_init(&fullA[s], 1);
      ptx::mbar_init(&emptyA[s], 1);
    }
    for (int s = 0; s < (p.b_stages < MAX_B_STAGES ? p.b_stages : MAX_B_STAGES); ++s) {
      ptx::mbar_init(&fullB[s], 1);
      ptx::mbar_init(&emptyB[s], 1);
    }
    for (int a = 0; a < MAX_SLOTS; ++a) {
      ptx::mbar_init(&tfull[a], 1);
      ptx::mbar_init(&tempty[a], PAIR ? 8 : 4);   // the four epilogue warps of one half-tile (of both CTAs)
    }
    ptx::fence_barrier_init();
  }
  if (PAIR) ptx::cluster_sync_all();             // both CTAs' barriers exist before anything arrives on them remotely
  if (warp == 2) {
    if (PAIR) {
      ptx::tmem_alloc_pair(tmem_slot, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      SlabIter ia, ib;
      ia.init(p, cta0, cta_step);
      ib.init(p, cta0, cta_step);
      const uint32_t txm = PAIR ? 2u : 1u;       // both CTAs' bytes land on the leader's barrier
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      auto issue_a = [&]() {
        const int s = sa;
        const uint32_t ph = pha;
        if (++sa == p.a_stages) { sa = 0; pha ^= 1; }
        int nb, w0, h0, n;
        tile_coords<PAIR>(p, ia.tile, rank, nb, w0, h0, n);
        const bool halo = p.taps[ia.seg] == 9;
        ptx::mbar_wait_backoff(&emptyA[s], ph ^ 1);
        if (rank == 0) ptx::mbar_arrive_expect_tx(&fullA[s], txm * (halo ? A_HALO_TX : A_PLAIN_BYTES));
        const CUtensorMap* mA = ia.seg ? &tmA1 : &tmA0;
        if (halo)
          ptx::load_4d<PAIR>(smA + s * A_HALO_BYTES, mA, &fullA[s], ia.kc * BLOCK_K, w0 - 1, h0 - 1, n);
        else
          ptx::load_4d<PAIR>(smA + s * A_HALO_BYTES, mA, &fullA[s], ia.kc * BLOCK_K, w0, h0, n);
        ia.next(p);
      };
      if (p.resident) {
        // the weights of a 64-output-channel layer fit in shared memory: fetch them once, then stream only A tiles
        const int slabs = p.C[0] / BLOCK_K;
        if (rank == 0) ptx::mbar_arrive_expect_tx(&fullB[0], txm * (uint32_t)(slabs * 9 * b_bytes));
        for (int kc = 0; kc < slabs; ++kc)
          for (int tap = 0; tap < 9; ++tap)
            ptx::load_2d<PAIR>(smB + (kc * 9 + tap) * b_bytes, &tmB0, &fullB[0], tap * p.C[0] + kc * BLOCK_K, rank * bn_cta);
        while (ia.valid) issue_a();
      }
      if (!p.resident && ia.valid) issue_a();
      while (!p.resident && ib.valid) {
        int nb, w0, h0, n;
        tile_coords<PAIR>(p, ib.tile, rank, nb, w0, h0, n);
        const int taps = p.taps[ib.seg];
        const int tps = taps == 9 ? p.tps : 1;
        const int look = taps - 1 < LOOKAHEAD_TAP ? taps - 1 : LOOKAHEAD_TAP;
        const CUtensorMap* mB = ib.seg ? &tmB1 : &tmB0;
        for (int tap0 = 0; tap0 < taps; tap0 += tps) {
          const int s = sb;
          const uint32_t ph = phb;
          if (++sb == p.b_stages) { sb = 0; phb ^= 1; }
          ptx::mbar_wait_backoff(&emptyB[s], ph ^ 1);
          if (rank == 0) ptx::mbar_arrive_expect_tx(&fullB[s], txm * (uint32_t)(b_bytes * tps));
          for (int j = 0; j < tps; ++j)
            ptx::load_2d<PAIR>(smB + s * bs_bytes + j * b_bytes, mB, &fullB[s], (tap0 + j) * p.C[ib.seg] + ib.kc * BLOCK_K,
                               nb * p.block_n + rank * bn_cta);
          if (tap0 <= look && look < tap0 + tps && ia.valid) issue_a();
        }
        ib.next(p);
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ============================== MMA issuer (PAIR: the leader CTA only) ==============================
    // The whole warp walks the schedule (uniform control flow, barrier waits by all lanes); one elected lane issues
    // the tcgen05 instructions.  The per-tap body is kept to a few dozen instructions: descriptor halves are
    // precomputed, ring indices wrap by compare instead of modulo -- the issuing thread, not the tensor pipe, was the
    // bottleneck of the first version (ncu: ~1190 cycles of scalar code per tap, profiles/r01_b_*).
    const uint32_t idesc = ptx::make_idesc_bf16(PAIR ? 2 * BLOCK_M : BLOCK_M, p.block_n, 0, 0);
    const uint32_t fullA_s = ptx::smem_u32(fullA), emptyA_s = ptx::smem_u32(emptyA);
    const uint32_t fullB_s = ptx::smem_u32(fullB), emptyB_s = ptx::smem_u32(emptyB);
    const uint32_t smA_s = ptx::smem_u32(smA), smB_s = ptx::smem_u32(smB);
    const uint32_t b_hi = ptx::desc_hi(1024);
    const uint32_t b_step = (uint32_t)b_bytes >> 4;
    SlabIter it;
    it.init(p, cta0, cta_step);
    int sa = 0, sb = 0, t = 0;
    uint32_t pha = 0, phb = 0;
    bool bres_ready = false;
    while (it.valid) {
      // half-tiles 2t (left) and 2t+1 (right) of this CTA's t-th tile: accumulator slots and their use counts
      const int sl = (2 * t) & p.slot_mask, sr = (2 * t + 1) & p.slot_mask;
      const uint32_t use_par = (uint32_t)((2 * t) >> p.slot_shift) & 1u;
      ptx::bar_wait_remote<PAIR>(&tempty[sl], use_par ^ 1);
      ptx::bar_wait_remote<PAIR>(&tempty[sr], use_par ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_l = tmem_base + (uint32_t)(sl * p.block_n), d_r = tmem_base + (uint32_t)(sr * p.block_n);
      const int cur_tile = it.tile;
      uint32_t accumulate = 0;
      while (it.valid && it.tile == cur_tile) {
        ptx::mbar_wait_s(fullA_s + sa * 8, pha);
        ptx::tc_fence_after();
        const int taps = p.taps[it.seg];
        const bool halo = taps == 9;
        const uint32_t a_hi = ptx::desc_hi(halo ? HALO_W * 128 : TILE_W * 128);
        const uint32_t a_lo0 = ptx::desc_lo(smA_s + sa * A_HALO_BYTES, 16);
        const int rem = p.C[it.seg] - it.kc * BLOCK_K;
        const int ksteps = rem >= BLOCK_K ? 4 : (rem + 15) / 16;   // channels past C are TMA zero fill
        // halo origin is pixel (h0-1, w0-1): tap (dy,dx) starts dy halo rows (3072 B) down and dx pixels (128 B) right;
        // the right half-tile starts 8 pixels (1024 B) further
        if (p.resident) {
          // 72 MMAs per slab straight from the resident weights: one barrier wait (the A tile) per 72 instructions
          if (!bres_ready) {
            ptx::mbar_wait_s(fullB_s, 0);
            ptx::tc_fence_after();
            bres_ready = true;
          }
          if (ptx::elect_one()) {
            const uint32_t b_lo = ptx::desc_lo(smB_s, 16) + it.kc * (9 * b_step);
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
              for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint64_t bd = ptx::pack_desc(b_lo + (dy * 3 + dx) * b_step + 2 * k, b_hi);
                  const uint32_t al = a_lo0 + dy * ROW_OFF + dx * 8 + 2 * k;
                  const uint32_t acc = (dy | dx | k) ? 1u : accumulate;
                  ptx::mma<PAIR>(d_l, ptx::pack_desc(al, a_hi), bd, idesc, acc);
                  ptx::mma<PAIR>(d_r, ptx::pack_desc(al + HALF_OFF, a_hi), bd, idesc, acc);
                }
          }
          accumulate = 1;
          __syncwarp();
        } else if (halo && p.tps == 3 && ksteps == 4) {
          // one kernel row (3 taps x 2 halves x 4 K-steps = 24 MMAs) per B stage, fully unrolled with immediate offsets
          uint32_t a_row = a_lo0;
          for (int dy = 0; dy < 3; ++dy) {
            ptx::mbar_wait_s(fullB_s + sb * 8, phb);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint32_t b_lo = ptx::desc_lo(smB_s, 16) + sb * (3 * b_step);
#pragma unroll
              for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint64_t bd = ptx::pack_desc(b_lo + dx * b_step + 2 * k, b_hi);
                  const uint32_t acc = (dx | k) ? 1u : accumulate;
                  ptx::mma<PAIR>(d_l, ptx::pack_desc(a_row + dx * 8 + 2 * k, a_hi), bd, idesc, acc);
                  ptx::mma<PAIR>(d_r, ptx::pack_desc(a_row + HALF_OFF + dx * 8 + 2 * k, a_hi), bd, idesc, acc);
                }
              }
              ptx::commit_s<PAIR>(emptyB_s + sb * 8);
            }
            accumulate = 1;
            __syncwarp();
            if (++sb == p.b_stages) { sb = 0; phb ^= 1; }
            a_row += ROW_OFF;
          }
        } else {
          const int tps = halo ? p.tps : 1;
          uint32_t a_row = a_lo0, a_lo = a_lo0;
          int dx = 0, j = 0;
          for (int tap = 0; tap < taps; ++tap) {
            if (j == 0) {
              ptx::mbar_wait_s(fullB_s + sb * 8, phb);
              ptx::tc_fence_after();
            }
            if (ptx::elect_one()) {
              const uint32_t b_lo = ptx::desc_lo(smB_s, 16) + sb * (p.tps * b_step) + j * b_step;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if (k < ksteps) {
                  const uint64_t bd = ptx::pack_desc(b_lo + 2 * k, b_hi);
                  ptx::mma<PAIR>(d_l, ptx::pack_desc(a_lo + 2 * k, a_hi), bd, idesc, accumulate);
                  ptx::mma<PAIR>(d_r, ptx::pack_desc(a_lo + HALF_OFF + 2 * k, a_hi), bd, idesc, accumulate);
                  accumulate = 1;
                }
              }
              if (j == tps - 1) ptx::commit_s<PAIR>(emptyB_s + sb * 8);
            }
            accumulate = 1;
            __syncwarp();
            if (++j == tps) {
              j = 0;
              if (++sb == p.b_stages) { sb = 0; phb ^= 1; }
            }
            if (++dx == 3) { dx = 0; a_row += ROW_OFF; a_lo = a_row; } else { a_lo += 128 >> 4; }
          }
        }
        if (ptx::elect_one()) ptx::commit_s<PAIR>(emptyA_s + sa * 8);
        __syncwarp();
        if (++sa == p.a_stages) { sa = 0; pha ^= 1; }
        it.next(p);
      }
      if (ptx::elect_one()) {
        ptx::commit_s<PAIR>(ptx::smem_u32(&tfull[sl]));
        ptx::commit_s<PAIR>(ptx::smem_u32(&tfull[sr]));
      }
      __syncwarp();
      ++t;
    }
  } else if (warp >= 2) {
    // ============================== epilogue (warps 2..9) ==============================
    // Warps 2-5 (half 0) drain the left 16 x 8-pixel half-tile of every tile, warps 6-9 the right one: accumulator row
    // r = 32 lg + lane is pixel (r >> 3, 8 half + (r & 7)) of the tile, and the warp drains all of its 32-column chunks.
    const int lg = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = lg * 32 + lane;
    const int hl = row >> 3, wl = HALF_W * half + (row & 7);
    EpiOut eo;
    eo.stat_acc = p.stats ? stat_smem + (warp - 2) * (EPI_STAT_CHUNKS * 64) : nullptr;
    eo.y = p.y; eo.y_ld = p.y_ld; eo.bias = p.bias; eo.scale = p.scale; eo.relu = p.relu; eo.addend = p.addend; eo.addend_ld = p.addend_ld;
    eo.Ncols = p.Ncols; eo.scatter = 0; eo.Cout = p.Ncols; eo.H = p.H; eo.W = p.W;
    const int mode = (p.addend ? 1 : 0) | (p.bias ? 2 : 0) | ((p.scale || p.relu) ? 4 : 0);
    // Staged stores: the warp's 32 accumulator rows are the 4 x 8 pixels (h0 + 4 lg .., w0 + 8 half ..) of the tile.  A
    // 64-column "job" (two 32-column chunks) is written to a SWIZZLE_128B buffer -- row = lane, 16-byte piece g at
    // (g ^ (lane & 7)) -- and leaves as ONE TMA box, which also clips ragged image edges.  The per-thread path stores
    // 16 bytes per lane at a 2 * y_ld byte pitch: 32 L1 wavefronts per instruction on the data pipe the tensor core
    // fetches its operands through (ncu: LSU wavefronts 25-46 % next to 63-73 % operand wavefronts).
    const uint32_t stg_s = ptx::smem_u32(stg_base + (warp - 2) * p.st_bufs * STG_BYTES);
    const uint32_t row_s = stg_s + (uint32_t)lane * 128u;
    const uint32_t sx = (uint32_t)lane & 7u;
    uint32_t job = 0;     // stores issued by this warp (staging buffer parity)
    // per-CTA BatchNorm statistics on the staged path (p.stats): sum / sum of squares per channel pair (lane) and 64-column
    // job, kept in registers for the life of the CTA -- all its tiles share one column block
    float sacc[4][4];
#pragma unroll
    for (int J = 0; J < 4; ++J) sacc[J][0] = sacc[J][1] = sacc[J][2] = sacc[J][3] = 0.f;
    auto locate = [&](int tile, int& nb, bool& valid, long long& pix, int& n, int& h, int& w) {
      int w0, h0;
      const bool ok = tile_coords<PAIR>(p, tile, rank, nb, w0, h0, n);
      h = h0 + hl;
      w = w0 + wl;
      valid = ok && h < p.H && w < p.W;
      pix = ((long long)n * p.H + h) * p.W + w;
    };
    int k = 0;
    int jc = 0;      // tile-statistics exchanges so far (buffer parity)
    int nb, n, h, w;
    bool valid;
    long long pix;
    uint4 ad[4];
    if (cta0 < p.total_tiles) {
      locate(cta0, nb, valid, pix, n, h, w);
      epi_prefetch(eo, nb * p.block_n, valid, pix, ad);
    }
    for (int tile = cta0; tile < p.total_tiles; tile += cta_step, ++k) {
      const int t = 2 * k + half;                 // half-tile counter of this CTA
      const int slot = t & p.slot_mask;
      const uint32_t par = (uint32_t)(t >> p.slot_shift) & 1u;
      int nb2 = 0, n2 = 0, h2 = 0, w2 = 0;
      bool valid2 = false;
      long long pix2 = 0;
      const bool more = tile + cta_step < p.total_tiles;
      if (more) locate(tile + cta_step, nb2, valid2, pix2, n2, h2, w2);
      ptx::mbar_wait(&tfull[slot], par);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(slot * p.block_n);
      bf16* yrow = p.y + pix * p.y_ld;
      // statistics chunk of this half-tile inside its image
      const int chunks_img = p.tiles_w * p.tiles_h * 2;
      const int tchunk = ((h - hl) / TILE_H * p.tiles_w + (w - wl) / TILE_W) * 2 + half;
      // tile statistics, second half: the four lane-group warps of this half-tile meet at a named barrier and warp lg == 0
      // writes one row per statistic for the 32 columns from col32 -- the [n][chunk][4][C] layout rbu_bn_stats' second
      // stage consumes
      auto combine_and_write = [&](const float* xb, int col32) {
        asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");
        if (lg == 0 && (!PAIR || n < p.N)) {
          float acc[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[q] = xb[q * 32 + lane];
#pragma unroll
          for (int g2 = 1; g2 < 4; ++g2) {
            acc[0] += xb[(g2 * 4 + 0) * 32 + lane];
            acc[1] += xb[(g2 * 4 + 1) * 32 + lane];
            acc[2] = fmaxf(acc[2], xb[(g2 * 4 + 2) * 32 + lane]);
            acc[3] = fminf(acc[3], xb[(g2 * 4 + 3) * 32 + lane]);
          }
          float* dstp = p.tile_stats + (((long long)n * chunks_img + tchunk) * 4) * p.Ncols + col32 + lane;
#pragma unroll
          for (int q = 0; q < 4; ++q) dstp[(long long)q * p.Ncols] = acc[q];
        }
      };
      // staged job (64 columns from jcol, or 32 for a trailing / clipped half) complete in this warp's buffer: hand the box
      // to the TMA store engine, then read the tile statistics off the staged bf16 values -- lane = channel pair, one
      // conflict-free 4-byte shared-memory load per pixel row instead of 31 shuffles per statistic and 32 columns
      auto finish_job = [&](int jcol, int chunks32) {
        const uint32_t jb = stg_s + ((p.st_bufs == 2 && (job & 1u)) ? (uint32_t)STG_BYTES : 0u);
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {   // lane 0 is the box origin: pixel (h0 + 4 lg, w0 + 8 half); columns past Ncols, pixels past the
                           // image and the tile of a pair's idle CTA (n >= N) are clipped by the tensor map
          ptx::tma_store_4d_s(&tmY, jb, jcol, w, h, n);
          ptx::bulk_commit();
        }
        ++job;
        if (p.tile_stats) {
          const unsigned rowmask = __ballot_sync(0xffffffffu, valid);    // lane r owns pixel row r of the box
          const uint32_t coff = ((uint32_t)lane & 3u) << 2, cch = (uint32_t)lane >> 2;
          float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f, mx0 = -INFINITY, mx1 = -INFINITY, mn0 = INFINITY, mn1 = INFINITY;
#pragma unroll
          for (int rr = 0; rr < 32; ++rr) {
            const uint32_t v2 = ptx::ld_shared_b32(jb + (uint32_t)rr * 128u + ((cch ^ ((uint32_t)rr & 7u)) << 4) + coff);
            if ((rowmask >> rr) & 1u) {
              const float f0 = __uint_as_float(v2 << 16), f1 = __uint_as_float(v2 & 0xffff0000u);
              s0 += f0; q0 += f0 * f0; mx0 = fmaxf(mx0, f0); mn0 = fminf(mn0, f0);
              s1 += f1; q1 += f1 * f1; mx1 = fmaxf(mx1, f1); mn1 = fminf(mn1, f1);
            }
          }
          for (int rd = 0; rd < chunks32; ++rd) {     // lanes 0-15 hold columns 0-31 of the job, lanes 16-31 columns 32-63
            float* xb = stat_smem + ((jc & 1) * 2 + half) * (4 * 4 * 32);     // [parity][half][lg][q][32]
            ++jc;
            if ((lane >> 4) == rd) {
              float* xw = xb + lg * (4 * 32) + 2 * (lane & 15);
              *reinterpret_cast<float2*>(xw) = make_float2(s0, s1);
              *reinterpret_cast<float2*>(xw + 32) = make_float2(q0, q1);
              *reinterpret_cast<float2*>(xw + 64) = make_float2(mx0, mx1);
              *reinterpret_cast<float2*>(xw + 96) = make_float2(mn0, mn1);
            }
            combine_and_write(xb, jcol + 32 * rd);
          }
        }
        if (p.stats) {
          const unsigned rowmask = __ballot_sync(0xffffffffu, valid);
          const uint32_t ja = jb + (((uint32_t)lane & 3u) << 2), cch = (uint32_t)lane >> 2;
          float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
          for (int rr = 0; rr < 32; ++rr) {
            const uint32_t v2 = ptx::ld_shared_b32(ja + (uint32_t)rr * 128u + ((cch ^ ((uint32_t)rr & 7u)) << 4));
            if ((rowmask >> rr) & 1u) {
              const float f0 = __uint_as_float(v2 << 16), f1 = __uint_as_float(v2 & 0xffff0000u);
              s0 += f0; q0 += f0 * f0;
              s1 += f1; q1 += f1 * f1;
            }
          }
          const int jj = (jcol - nb * p.block_n) >> 6;
#pragma unroll
          for (int J = 0; J < 4; ++J)
            if (J == jj) { sacc[J][0] += s0; sacc[J][1] += s1; sacc[J][2] += q0; sacc[J][3] += q1; }
        }
      };
      for (int c0 = 0; c0 < p.block_n; c0 += 32) {
        const int col = nb * p.block_n + c0;
        if (p.tma_store && col >= p.Ncols) {
          // chunk past the last output column (Ncols % 32 == 0 here): nothing to compute, but a first half waiting in
          // the staging buffer still has to leave
          if (c0 & 32) finish_job(col - 32, 1);
        } else if ((p.stats && !p.tma_store) || col + 32 > p.Ncols) {
          epi_finish(eo, t_addr + (uint32_t)c0, col, valid, pix, n, h, w, ad, c0 >> 5);
        } else {
          uint32_t r[32];
          ptx::tmem_ld_32x32(t_addr + (uint32_t)c0, r);
          ptx::tmem_ld_wait();
          uint4 out[4];
          switch (mode) {   // warp-uniform: one lean arithmetic body per combination
            case 0: epi_math<false, false, false>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 1: epi_math<true, false, false>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 2: epi_math<false, true, false>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 3: epi_math<true, true, false>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 4: epi_math<false, false, true>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 5: epi_math<true, false, true>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            case 6: epi_math<false, true, true>(r, p.bias, p.scale, p.relu, col, ad, out); break;
            default: epi_math<true, true, true>(r, p.bias, p.scale, p.relu, col, ad, out); break;
          }
          if (p.tma_store) {
            const bool first = (c0 & 32) == 0;
            const uint32_t buf = row_s + ((p.st_bufs == 2 && (job & 1u)) ? (uint32_t)STG_BYTES : 0u);
            if (first) {   // the store that last read this buffer has drained it
              if (lane == 0) {
                if (p.st_bufs == 2) ptx::bulk_wait_read<1>(); else ptx::bulk_wait_read<0>();
              }
              __syncwarp();
            }
            const uint32_t pb = first ? 0u : 4u;
#pragma unroll
            for (int g = 0; g < 4; ++g) ptx::st_shared_v4(buf + (((pb + (uint32_t)g) ^ sx) << 4), out[g]);
            if (!first) finish_job(col - 32, 2);
            else if (c0 + 32 >= p.block_n) finish_job(col, 1);
          } else if (valid) {
            uint4* dst = reinterpret_cast<uint4*>(yrow + col);
            dst[0] = out[0]; dst[1] = out[1]; dst[2] = out[2]; dst[3] = out[3];
          }
          if (p.tile_stats && !p.tma_store) {
            // per-thread-store path: the warp reduces its 32 pixels per column with shuffles (lane l ends up with column l),
            // then the same exchange as the staged path
            float rv[32], tmp[32];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              bf16x8 t8;
              *reinterpret_cast<uint4*>(&t8) = out[g];
              unpack8(t8, &rv[g * 8]);
            }
            float red[4];
#pragma unroll
            for (int i = 0; i < 32; ++i) tmp[i] = valid ? rv[i] : 0.f;
            red[0] = warp_colsum32(tmp, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i) tmp[i] = valid ? rv[i] * rv[i] : 0.f;
            red[1] = warp_colsum32(tmp, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i) tmp[i] = valid ? rv[i] : -INFINITY;
            red[2] = warp_colext32<true>(tmp, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i) tmp[i] = valid ? rv[i] : INFINITY;
            red[3] = warp_colext32<false>(tmp, lane);
            float* xb = stat_smem + ((jc & 1) * 2 + half) * (4 * 4 * 32);     // [parity][half][lg][q][32]
            ++jc;
#pragma unroll
            for (int q = 0; q < 4; ++q) xb[(lg * 4 + q) * 32 + lane] = red[q];
            combine_and_write(xb, col);
          }
        }
        if (c0 + 32 < p.block_n)
          epi_prefetch(eo, col + 32, valid, pix, ad);
        else if (more)
          epi_prefetch(eo, nb2 * p.block_n, valid2, pix2, ad);   // next tile
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) ptx::mbar_arrive_cluster(&tempty[slot], 0); else ptx::mbar_arrive(&tempty[slot]);
      }
      nb = nb2; n = n2; h = h2; w = w2; valid = valid2; pix = pix2;
    }
    if (p.tma_store && lane == 0) ptx::bulk_wait_read<0>();   // shared memory stays allocated until the last box is read
    if (p.stats && p.tma_store) {
      // every tile of this CTA (pair) has the same column block: the eight epilogue warps park their register accumulators
      // in their drained staging buffers -- [job][lane] x (s0, s1, q0, q1) -- and warp J adds the eight up in warp order:
      // ONE row [2][Ncols] per CTA
      __syncwarp();
#pragma unroll
      for (int J = 0; J < 4; ++J)
        ptx::st_shared_v4(stg_s + (uint32_t)((J * 32 + lane) * 16),
                          make_uint4(__float_as_uint(sacc[J][0]), __float_as_uint(sacc[J][1]), __float_as_uint(sacc[J][2]),
                                     __float_as_uint(sacc[J][3])));
      asm volatile("bar.sync 3, 256;" ::: "memory");
      const int J = warp - 2;
      const int nbf = cta0 % p.n_blocks;
      const int col = nbf * p.block_n + J * 64 + 2 * lane;
      if (J < 4 && J * 64 < p.block_n && col < p.Ncols) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const uint32_t base0 = ptx::smem_u32(stg_base) + (uint32_t)((J * 32 + lane) * 16);
        for (int w8 = 0; w8 < 8; ++w8) {
          const uint4 v = ptx::ld_shared_v4(base0 + (uint32_t)(w8 * p.st_bufs * STG_BYTES));
          a0 += __uint_as_float(v.x); a1 += __uint_as_float(v.y); a2 += __uint_as_float(v.z); a3 += __uint_as_float(v.w);
        }
        float* row_out = p.stats + (long long)blockIdx.x * 2 * p.Ncols;
        *reinterpret_cast<float2*>(row_out + col) = make_float2(a0, a1);
        *reinterpret_cast<float2*>(row_out + p.Ncols + col) = make_float2(a2, a3);
      }
    } else if (p.stats) {
      // per-thread-store path: the eight epilogue warps' shared-memory accumulators are added up in warp order and leave as
      // ONE row per CTA (warp j flushes the 32-column chunk j)
      asm volatile("bar.sync 3, 256;" ::: "memory");
      const int nbf = cta0 % p.n_blocks;
      const int j = warp - 2;
      const int col = nbf * p.block_n + j * 32 + lane;
      if (j * 32 < p.block_n && col < p.Ncols) {
        float2 acc = make_float2(0.f, 0.f);
        for (int w8 = 0; w8 < 8; ++w8) {
          const float2 v = reinterpret_cast<const float2*>(stat_smem + w8 * (EPI_STAT_CHUNKS * 64))[j * 32 + lane];
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
  if (PAIR) {
    __syncwarp();
    ptx::cluster_sync_all();                     // neither CTA may leave (or free TMEM) while its peer still uses the pair
    if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, (uint32_t)p.tmem_cols);
  } else {
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmB0,
                 const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
                 const __grid_constant__ CUtensorMap tmY, const __grid_constant__ HParams p) {
  conv_halo_body<false>(tmA0, tmB0, tmA1, tmB1, tmY, p);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_halo_pair_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmB0,
                      const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
                      const __grid_constant__ CUtensorMap tmY, const __grid_constant__ HParams p) {
  conv_halo_body<true>(tmA0, tmB0, tmA1, tmB1, tmY, p);
}

}  // namespace

// Returns 1 if the halo kernel can run these arguments (3x3 dilation-1 and 1x1 segments on images of at least
// 16 x 16 pixels, no gather / scatter), else 0.
int rbu_conv_halo_supported(const rbu_conv_gemm_args* a) {
  if (a->scatter || a->H < TILE_H || a->W < TILE_W) return 0;
  // per-CTA statistics: register accumulators on the staged path (any width that is whole 32-column chunks), shared-memory
  // accumulators covering 128 columns on the per-thread path
  if (a->stats && a->Ncols > 32 * EPI_STAT_CHUNKS && a->Ncols % 32 != 0) return 0;
  int any3x3 = 0;
  for (int s = 0; s < a->nseg; ++s) {
    const rbu_gemm_operand& o = a->seg[s];
    if (o.gather) return 0;
    if (!(o.taps == 1 || (o.taps == 9 && o.dil == 1))) return 0;
    any3x3 |= o.taps == 9;
  }
  return any3x3;   // pure 1x1 GEMMs have no halo to reuse: the generic kernel's deeper A+B ring is faster for them
}

// Argument validation is done by the caller (rbu_conv_gemm).
int rbu_conv_halo_launch(const rbu_conv_gemm_args* a, cudaStream_t stream) {
  HParams p;
  memset(&p, 0, sizeof(p));
  p.N = a->N; p.H = a->H; p.W = a->W;
  p.tiles_w = rbu_cdiv(a->W, TILE_W);
  p.tiles_h = rbu_cdiv(a->H, TILE_H);
  p.Ncols = a->Ncols;
  // 128-column blocks from 128 output channels up: four accumulator slots (two tiles in flight), so the epilogue of one
  // tile always overlaps the MMAs of the next -- with 256-column blocks the two half-tiles fill the TMEM and the MMA
  // issuer waited 40% of the time for the drain (ncu, 256->256 at 64x64: 1438 vs 1480 TFLOP/s).  One-tile images
  // (16 x 16, 1024 channels) keep 256: half as many activation re-reads per weight block (1503 vs 1393 TFLOP/s).
  const bool one_tile = p.tiles_w * p.tiles_h == 1;
  p.block_n = a->Ncols >= 256 ? (one_tile ? 256 : 128) : (a->Ncols >= 128 ? 128 : ((a->Ncols + 31) / 32) * 32);
  p.n_blocks = rbu_cdiv(a->Ncols, p.block_n);
  p.fd_nb = make_fastdiv(p.n_blocks);
  p.fd_tw = make_fastdiv(p.tiles_w);
  p.fd_th = make_fastdiv(p.tiles_h);
  p.slot_shift = 4 * p.block_n <= 512 ? 2 : 1;
  p.slot_mask = (1 << p.slot_shift) - 1;
  p.nseg = a->nseg;
  for (int s = 0; s < a->nseg; ++s) {
    p.taps[s] = a->seg[s].taps;
    p.C[s] = a->seg[s].C;
  }
  // CTA pairs (cta_group::2) halve the weight bytes every SM pulls from L2 -- what bounded the >= 128-channel layers --
  // and make the 128->64 layer's weights resident (72 KB per CTA).  Not used where a single CTA already keeps the whole
  // weight operand resident (64->64: nothing left to halve, and the pair's lock step costs 10 %; measured 918 vs 1020
  // TFLOP/s), with the per-CTA output statistics (unused by the engine), or for column blocks whose halves are not whole
  // 8-row swizzle groups.
  const bool single_resident = a->nseg == 1 && a->seg[0].taps == 9 && p.n_blocks == 1 && a->seg[0].C % BLOCK_K == 0 &&
                               (long)(a->seg[0].C / BLOCK_K) * 9 * p.block_n * 128 + 2 * A_HALO_BYTES <= SMEM_LIMIT - 2048;
  const bool pair = !single_resident && p.block_n % 32 == 0 && rbu_num_sms() >= 2 &&
                    (!a->stats || p.n_blocks <= rbu_num_sms() / 2);
  const int b_bytes = (pair ? p.block_n / 2 : p.block_n) * 128;     // one tap's weight tile in ONE CTA's shared memory
  p.tps = p.block_n <= 128 ? 3 : 1;
  p.a_stages = 2;
  // Staged epilogue (TMA stores) when the output is whole 32-column chunks and the staging buffers (8 warps x 4 KB, two per
  // warp if the weight ring keeps >= 3 stages) fit.
  const bool can_stage = a->Ncols % 32 == 0 && ((uintptr_t)a->y & 15) == 0 && a->y_ld % 8 == 0;
  const int ring_room = SMEM_LIMIT - 2048 - p.a_stages * A_HALO_BYTES;
  p.tma_store = 0;
  p.st_bufs = 0;
  if (can_stage) {
    for (int bufs = 2; bufs >= 1 && !p.tma_store; --bufs)
      if ((ring_room - 8 * bufs * STG_BYTES) / (b_bytes * p.tps) >= (bufs == 2 ? 3 : 2)) {
        p.tma_store = 1;
        p.st_bufs = bufs;
      }
  }
  p.b_stages = (ring_room - 8 * p.st_bufs * STG_BYTES) / (b_bytes * p.tps);
  if (p.b_stages > MAX_B_STAGES) p.b_stages = MAX_B_STAGES;
  {
    // resident weights: one 3x3 segment, one column block, whole operand <= the shared memory left beside 2-3 A stages
    const long wbytes = (long)(a->seg[0].C / BLOCK_K) * 9 * b_bytes;
    if (a->nseg == 1 && a->seg[0].taps == 9 && p.n_blocks == 1 && a->seg[0].C % BLOCK_K == 0) {
      const int as = 2;   // a third stage does not help (pair 64->64: 759 vs 918 TFLOP/s)
      if (wbytes + as * A_HALO_BYTES <= SMEM_LIMIT - 2048) {
        const long room = SMEM_LIMIT - 2048 - wbytes - as * A_HALO_BYTES;
        p.st_bufs = can_stage ? (room >= 16 * STG_BYTES ? 2 : (room >= 8 * STG_BYTES ? 1 : 0)) : 0;
        p.tma_store = p.st_bufs > 0;
        p.resident = 1;
        p.a_stages = as;
        p.tps = 1;
        p.b_stages = (int)(wbytes / b_bytes);       // the B region is sized in single-tap tiles
      }
    }
  }
  p.tmem_cols = 32;
  while (p.tmem_cols < (p.slot_mask + 1) * p.block_n) p.tmem_cols <<= 1;
  p.sp_total = p.tiles_w * p.tiles_h * a->N;
  p.total_tiles = (pair ? (p.sp_total + 1) / 2 : p.sp_total) * p.n_blocks;
  p.y = reinterpret_cast<bf16*>(a->y);
  p.y_ld = a->y_ld;
  p.bias = a->bias;
  p.scale = a->scale;
  p.relu = a->relu;
  p.addend = reinterpret_cast<const bf16*>(a->addend);
  p.addend_ld = a->addend_ld;
  p.stats = a->stats;
  p.tile_stats = a->tile_stats;
  if (a->tile_stats)
    RBU_CHECK_ARG(!a->stats && a->Ncols % 32 == 0 && ((uintptr_t)a->tile_stats & 15) == 0,
                  "rbu_conv_gemm: tile statistics need Ncols %% 32 == 0 and exclude the per-CTA statistics");

  CUtensorMap tmA[2], tmB[2];
  memset(tmA, 0, sizeof(tmA));
  memset(tmB, 0, sizeof(tmB));
  for (int s = 0; s < a->nseg; ++s) {
    const rbu_gemm_operand& o = a->seg[s];
    const bool halo = o.taps == 9;
    const uint64_t dims[4] = {(uint64_t)o.C, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)o.x_ld * 2, (uint64_t)o.x_ld * 2 * a->W, (uint64_t)o.x_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {BLOCK_K, (uint32_t)(halo ? HALO_W : TILE_W), (uint32_t)(halo ? HALO_H : TILE_H), 1};
    int rc = rbu_encode_tmap_bf16(&tmA[s], o.x, 4, dims, str, box);
    if (rc) return rc;
    const uint64_t ktot = (uint64_t)o.taps * o.C;
    const uint64_t bdims[2] = {ktot, (uint64_t)a->Ncols};
    const uint64_t bstr[1] = {ktot * 2};
    const uint32_t bbox[2] = {BLOCK_K, (uint32_t)(pair ? p.block_n / 2 : p.block_n)};
    rc = rbu_encode_tmap_bf16(&tmB[s], o.w, 2, bdims, bstr, bbox);
    if (rc) return rc;
  }
  if (a->nseg == 1) {
    tmA[1] = tmA[0];
    tmB[1] = tmB[0];
  }
  CUtensorMap tmY;
  memset(&tmY, 0, sizeof(tmY));
  if (p.tma_store) {
    const uint64_t dims[4] = {(uint64_t)a->Ncols, (uint64_t)a->W, (uint64_t)a->H, (uint64_t)a->N};
    const uint64_t str[3] = {(uint64_t)a->y_ld * 2, (uint64_t)a->y_ld * 2 * a->W, (uint64_t)a->y_ld * 2 * a->W * a->H};
    const uint32_t box[4] = {64, HALF_W, 4, 1};
    const int rc = rbu_encode_tmap_bf16(&tmY, a->y, 4, dims, str, box);
    if (rc) return rc;
  }
  const int smem_bytes = p.a_stages * A_HALO_BYTES + p.b_stages * b_bytes * p.tps + 8 * p.st_bufs * STG_BYTES + 1024 + 512;
  static std::atomic<unsigned long long> attr_set{0};      // one bit per device ordinal
  if (rbu_first_use_on_device(&attr_set))
    RBU_CHECK_CUDA(cudaFuncSetAttribute(conv_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  if (pair) {
    static std::atomic<unsigned long long> attr_pair{0};
    if (rbu_first_use_on_device(&attr_pair))
      RBU_CHECK_CUDA(cudaFuncSetAttribute(conv_halo_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    int pairs = rbu_num_sms() / 2;
    if (pairs > p.total_tiles) pairs = p.total_tiles;
    if (a->stats) {
      pairs = pairs / p.n_blocks * p.n_blocks;     // every pair keeps one column block: work unit stride % n_blocks == 0
      RBU_CHECK_ARG(pairs > 0 && (p.tma_store || p.block_n <= 32 * EPI_STAT_CHUNKS) && ((uintptr_t)a->stats & 15) == 0,
                    "rbu_conv_gemm: output statistics are not supported for this shape");
      const size_t row_floats = (size_t)2 * a->Ncols, written = (p.tma_store && p.n_blocks == 1) ? (size_t)2 * pairs : 0;
      const size_t total = rbu_conv_stats_floats(a->Ncols);
      if (written * row_floats < total)
        RBU_CHECK_CUDA(cudaMemsetAsync(a->stats + written * row_floats, 0, (total - written * row_floats) * sizeof(float), stream));
    }
    const int gridp = 2 * pairs;
    conv_halo_pair_kernel<<<gridp, NUM_THREADS, smem_bytes, stream>>>(tmA[0], tmB[0], tmA[1], tmB[1], tmY, p);
    RBU_CHECK_LAUNCH();
    return RBU_OK;
  }
  int grid = p.total_tiles < rbu_num_sms() ? p.total_tiles : rbu_num_sms();
  if (a->stats) {
    grid = grid / p.n_blocks * p.n_blocks;         // every CTA keeps one column block
    RBU_CHECK_ARG(grid > 0 && (p.tma_store || p.block_n <= 32 * EPI_STAT_CHUNKS) && ((uintptr_t)a->stats & 15) == 0,
                  "rbu_conv_gemm: output statistics are not supported for this shape");
    const size_t row_floats = (size_t)2 * a->Ncols, written = (p.tma_store && p.n_blocks == 1) ? (size_t)grid : 0;
    const size_t total = rbu_conv_stats_floats(a->Ncols);
    if (written * row_floats < total)
      RBU_CHECK_CUDA(cudaMemsetAsync(a->stats + written * row_floats, 0, (total - written * row_floats) * sizeof(float), stream));
  }
  conv_halo_kernel<<<grid, NUM_THREADS, smem_bytes, stream>>>(tmA[0], tmB[0], tmA[1], tmB[1], tmY, p);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
