// Outer contours of water masks: cv2.findContours(mask, RETR_EXTERNAL, CHAIN_APPROX_NONE | CHAIN_APPROX_SIMPLE).
//
// Definition (include/rbunet.h, DESIGN.md §8 item 10).  Foreground components are 8-connected and the image is framed by
// background.  A component is traced iff the 4-connected background component (frame included) holding the pixel above
// its raster-first pixel p0 touches the frame.  Chain codes 0 = (+1,0), 1 = (+1,-1), 2 = (0,-1) ... 7 = (+1,+1), y down.
// From p0 the first foreground neighbour i1 among codes 4, 3, 2, 1, 0, 7, 6, 5 (none: the contour is p0 alone).  A state
// (p, c) has c pointing at the previous pixel; its successor scans c+1, c+2, ... around p for the first foreground
// neighbour q at code d and is (q, d^4).  The contour is the cycle of states from (p0, code of i1), one point per
// state; SIMPLE keeps a state whose outgoing code differs from its predecessor's (whose outgoing code is c^4).
// Contours come out in decreasing raster order of p0.
//
// Every state on a traced contour has a background neighbour at code c+1, so the states of a pixel are the codes c with
// foreground at c and background at c+1: at most 4 per pixel, and at most 8/3 (H*W + frame) per image (each maps to a
// distinct background pixel and direction).  They are numbered densely, per pixel block, in a deterministic order.
//   trace  fg union-find at 8 and bg union-find at 4 (the passes of components.cuh, three launches each);
//          frame: every bg root touching the image border gets FLAG;
//          nb:    per pixel the fg bit and the 8-neighbour fg mask, per block the state count;  scan;  base: per pixel
//                 the index of its first state;
//          links: per state the pixel (meta) and the 64-bit word (successor << 32 | weight); the start state of an
//                 external component is a root: (itself, successor); a successor that is no state ends a dead chain;
//          jump:  R = ceil(log2(capacity)) rounds of in-place pointer jumping on the packed words: a word always holds a
//                 state it reaches and the weight up to there, so concurrent updates only speed it up;
//          count: per pixel in decreasing raster order, 1 contour and K points at each external start (K = the root's
//                 weight + the jumped weight of its successor);  scan -> counts_out.
//   write  offsets: contour k's point offset; the root's word keeps its successor and takes the end of its points, and
//          the start point is written;  points: every kept state reaching a root writes at end - weight.  Repeatable.
// States of holes and of non-external components never reach a root and are dropped.  Integer arithmetic only, no
// atomics outside the union-find: the same bits run to run and for an image alone or inside a batch.
#include <algorithm>

#include "components.cuh"

namespace {

constexpr int PT = 256;                            // threads of the per-pixel passes
constexpr int PPT = 4;                             // pixels per thread
constexpr int PB = PT * PPT;                       // pixels per block
constexpr int SCAN_T = 1024;
constexpr int JUMP_T = 256;
constexpr int JUMP_MAX_CTAS = 2048;                // per image; the state passes loop over the rest
constexpr int FLAG = 1 << 30;                      // bg root touching the frame (indices are below 2^30)
constexpr unsigned ROOT = 1u << 31, KEEP = 1u << 30, PIX = KEEP - 1;

__constant__ int DX[8] = {1, 1, 0, -1, -1, -1, 0, 1};
__constant__ int DY[8] = {0, -1, -1, -1, 0, 1, 1, 1};

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

bool dims_ok(int B, int H, int W) { return B >= 1 && B <= 65535 && H >= 1 && W >= 1 && H <= 32768 && W <= 32768; }

struct Layout {
  size_t pfg, pbg, nb, base, sblk, stot, meta, link, cblk, ctot, total;
  long long cap;                                   // states per image
  int nblk, rounds;
};

Layout layout(int B, int H, int W) {
  Layout L;
  const long long HW = (long long)H * W;
  L.cap = std::min(4 * HW, 8 * (HW + 2LL * H + 2LL * W + 4) / 3);
  L.nblk = rbu_cdiv(HW, PB);
  L.rounds = 1;
  while ((1LL << L.rounds) < L.cap) ++L.rounds;
  const size_t n = (size_t)B * HW, nb = (size_t)B * L.nblk, ns = (size_t)B * L.cap;
  L.pfg = 0;
  L.pbg = align256(L.pfg + n * 4);
  L.nb = align256(L.pbg + n * 4);
  L.base = align256(L.nb + n * 2);
  L.sblk = align256(L.base + n * 4);
  L.stot = align256(L.sblk + nb * 8);
  L.meta = align256(L.stot + (size_t)B * 8);
  L.link = align256(L.meta + ns * 4);
  L.cblk = align256(L.link + ns * 8);
  L.ctot = align256(L.cblk + nb * 16);
  L.total = align256(L.ctot + (size_t)B * 16);
  return L;
}

struct Ws {
  int *pfg, *pbg;
  uint16_t* nb;
  unsigned* base;
  long long *sblk, *stot;
  unsigned* meta;
  unsigned long long* link;
  long long *cblk, *ctot;
};

Ws carve(void* ws, const Layout& L) {
  uint8_t* w = static_cast<uint8_t*>(ws);
  return {reinterpret_cast<int*>(w + L.pfg), reinterpret_cast<int*>(w + L.pbg), reinterpret_cast<uint16_t*>(w + L.nb),
          reinterpret_cast<unsigned*>(w + L.base), reinterpret_cast<long long*>(w + L.sblk),
          reinterpret_cast<long long*>(w + L.stot), reinterpret_cast<unsigned*>(w + L.meta),
          reinterpret_cast<unsigned long long*>(w + L.link), reinterpret_cast<long long*>(w + L.cblk),
          reinterpret_cast<long long*>(w + L.ctot)};
}

// The codes c of m (8-neighbour fg mask) with fg at c and bg at c+1.
__device__ __forceinline__ unsigned state_mask(unsigned m) { return m & ~((m >> 1) | (m << 7)) & 0xFFu; }

__device__ __forceinline__ int slot(unsigned sm, int c) { return __popc(sm & ((1u << c) - 1)); }

// The first fg code after c (c+1, ..., c+8); m has bit c set.
__device__ __forceinline__ int out_code(unsigned m, int c) {
  const unsigned r = ((m | (m << 8)) >> (c + 1)) & 0xFFu;
  return (c + __ffs(r)) & 7;
}

// The first fg code among 4, 3, 2, 1, 0, 7, 6, 5; m != 0.
__device__ __forceinline__ int start_code(unsigned m) {
  for (int k = 0; k < 8; ++k) {
    const int c = (12 - k) & 7;
    if ((m >> c) & 1) return c;
  }
  return -1;
}

// Exclusive scan over the block of NV int64 values per thread (thread order), with the block totals.
template <int NV, int WARPS>
__device__ __forceinline__ void block_scan(const long long (&v)[NV], long long (&excl)[NV], long long (&tot)[NV]) {
  __shared__ long long wsum[NV][WARPS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  long long inc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    inc[k] = v[k];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long n = __shfl_up_sync(0xffffffffu, inc[k], o);
      if (lane >= o) inc[k] += n;
    }
    if (lane == 31) wsum[k][w] = inc[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    long long before = 0, all = 0;
    for (int i = 0; i < WARPS; ++i) {
      const long long s = wsum[k][i];
      before += i < w ? s : 0;
      all += s;
    }
    excl[k] = before + inc[k] - v[k];
    tot[k] = all;
  }
  __syncthreads();                                   // wsum may be reused
}

// ------------------------------------------------------------------------------------------------ frame flags
// grid (ceil((2W + 2H) / 256), B): the bg root of every bg pixel on the image border gets FLAG.
__global__ void __launch_bounds__(256) ct_frame_kernel(int H, int W, int* __restrict__ pbg) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= 2 * (W + H)) return;
  int x, y;
  if (i < W) x = i, y = 0;
  else if (i < 2 * W) x = i - W, y = H - 1;
  else if (i < 2 * W + H) x = 0, y = i - 2 * W;
  else x = W - 1, y = i - 2 * W - H;
  int* P = pbg + (long long)blockIdx.y * H * W;
  const int v = P[y * W + x];
  if (v < 0) return;
  const int r = v & (FLAG - 1);
  P[r] = r | FLAG;                                    // every writer stores the same value
}

// ------------------------------------------------------------------------------------------------ states
// grid (nblk, B), PT threads; thread t owns pixels blk*PB + t*PPT .. +PPT-1.  nb[p] = fg << 8 | 8-neighbour fg mask;
// sblk[b][blk] = the block's state count.
__global__ void __launch_bounds__(PT)
ct_nb_kernel(int H, int W, int nblk, const int* __restrict__ pfg, uint16_t* __restrict__ nb, long long* __restrict__ sblk) {
  const long long off = (long long)blockIdx.y * H * W;
  const int HW = H * W;
  const int* P = pfg + off;
  long long cnt = 0;
  for (int j = 0; j < PPT; ++j) {
    const int p = blockIdx.x * PB + threadIdx.x * PPT + j;
    if (p >= HW) break;
    unsigned v = 0;
    if (P[p] >= 0) {
      const int x = p % W, y = p / W;
      unsigned m = 0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int xx = x + DX[c], yy = y + DY[c];
        if (xx >= 0 && xx < W && yy >= 0 && yy < H && P[yy * W + xx] >= 0) m |= 1u << c;
      }
      v = 0x100u | m;
      cnt += __popc(state_mask(m));
    }
    nb[off + p] = (uint16_t)v;
  }
  long long e[1], t[1];
  block_scan<1, PT / 32>({cnt}, e, t);
  if (threadIdx.x == 0) sblk[(long long)blockIdx.y * nblk + blockIdx.x] = t[0];
}

// grid B, SCAN_T threads: v[b][*] (NV values per entry) becomes its exclusive scan; tot[b][*] (and out[b][*] when
// given) the totals.
template <int NV>
__global__ void __launch_bounds__(SCAN_T)
ct_scan_kernel(int nblk, long long* __restrict__ v, long long* __restrict__ tot, long long* __restrict__ out) {
  long long* a = v + (long long)blockIdx.x * nblk * NV;
  long long carry[NV] = {};
  for (int base = 0; base < nblk; base += SCAN_T) {
    const int i = base + threadIdx.x;
    long long x[NV], e[NV], t[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) x[k] = i < nblk ? a[(long long)i * NV + k] : 0;
    block_scan<NV, SCAN_T / 32>(x, e, t);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (i < nblk) a[(long long)i * NV + k] = carry[k] + e[k];
      carry[k] += t[k];
    }
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      tot[blockIdx.x * NV + k] = carry[k];
      if (out) out[blockIdx.x * NV + k] = carry[k];
    }
  }
}

// grid (nblk, B): base[p] = the index of p's first state.
__global__ void __launch_bounds__(PT)
ct_base_kernel(int HW, int nblk, const uint16_t* __restrict__ nb, const long long* __restrict__ sblk,
               unsigned* __restrict__ base) {
  const long long off = (long long)blockIdx.y * HW;
  int c[PPT];
  long long cnt = 0;
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int p = blockIdx.x * PB + threadIdx.x * PPT + j;
    c[j] = p < HW ? __popc(state_mask(nb[off + p] & 0xFFu)) : 0;
    cnt += c[j];
  }
  long long e[1], t[1];
  block_scan<1, PT / 32>({cnt}, e, t);
  long long s = sblk[(long long)blockIdx.y * nblk + blockIdx.x] + e[0];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int p = blockIdx.x * PB + threadIdx.x * PPT + j;
    if (p < HW) base[off + p] = (unsigned)s;
    s += c[j];
  }
}

// Per-image views of the workspace.
struct Img {
  const int *pfg, *pbg;
  const uint16_t* nb;
  const unsigned* base;
  int H, W;
};

__device__ __forceinline__ Img img(const Ws& w, int b, int H, int W) {
  const long long off = (long long)b * H * W;
  return {w.pfg + off, w.pbg + off, w.nb + off, w.base + off, H, W};
}

// The successor state of (p, c) (c a state code of p), or -1 when (q, d^4) is no state of q.
__device__ __forceinline__ long long successor(const Img& I, int p, int c, int* dout) {
  const int d = out_code(I.nb[p] & 0xFFu, c);
  *dout = d;
  const int q = p + DX[d] + DY[d] * I.W, c2 = (d + 4) & 7;
  const unsigned sq = state_mask(I.nb[q] & 0xFFu);
  if (!((sq >> c2) & 1)) return -1;
  return (long long)I.base[q] + slot(sq, c2);
}

// Contour start at p: -1 when p starts no traced contour, -2 for a single point, else the start state s0.
__device__ __forceinline__ long long start_state(const Img& I, int p, int* c1) {
  if (I.pfg[p] != p) return -1;
  if (p >= I.W) {
    const int r = I.pbg[p - I.W] & (FLAG - 1);      // the pixel above p is background (p is raster-first)
    if (!(I.pbg[r] & FLAG)) return -1;
  }
  const unsigned m = I.nb[p] & 0xFFu;
  if (!m) return -2;
  *c1 = start_code(m);
  return (long long)I.base[p] + slot(state_mask(m), *c1);
}

// grid (nblk, B): every state's meta (pixel | KEEP | ROOT) and link word.
__global__ void __launch_bounds__(PT) ct_links_kernel(Ws w, int H, int W, long long cap, int approx) {
  const Img I = img(w, blockIdx.y, H, W);
  const long long so = (long long)blockIdx.y * cap;
  for (int j = 0; j < PPT; ++j) {
    const int p = blockIdx.x * PB + threadIdx.x * PPT + j;
    if (p >= H * W) break;
    unsigned sm = state_mask(I.nb[p] & 0xFFu);
    if (!sm) continue;
    int c1 = -1;
    const long long s0 = start_state(I, p, &c1);
    long long s = I.base[p];
    for (; sm; sm &= sm - 1, ++s) {
      const int c = __ffs(sm) - 1;
      int d;
      const long long n = successor(I, p, c, &d);
      const unsigned keep = approx == RBU_APPROX_NONE || d != (c ^ 4);
      const bool root = s == s0;
      w.meta[so + s] = (unsigned)p | (keep ? KEEP : 0u) | (root ? ROOT : 0u);
      unsigned long long word;
      if (root) word = (unsigned long long)s << 32 | (unsigned long long)n;     // n >= 0 on a traced contour
      else if (n < 0) word = (unsigned long long)s << 32;                       // a dead end: never reaches a root
      else word = (unsigned long long)n << 32 | keep;
      w.link[so + s] = word;
    }
  }
}

// grid (<= JUMP_MAX_CTAS, B): one round of pointer jumping over the image's states.
__global__ void __launch_bounds__(JUMP_T)
ct_jump_kernel(long long cap, const long long* __restrict__ stot, const unsigned* __restrict__ meta,
               unsigned long long* __restrict__ link) {
  const long long so = (long long)blockIdx.y * cap, n = stot[blockIdx.y];
  const unsigned* M = meta + so;
  unsigned long long* L = link + so;
  for (long long s = (long long)blockIdx.x * JUMP_T + threadIdx.x; s < n; s += (long long)gridDim.x * JUMP_T) {
    const unsigned long long a = __ldcg(L + s);
    const unsigned t = (unsigned)(a >> 32);
    if (M[t] & ROOT) continue;                       // done (roots point at themselves)
    const unsigned long long b = __ldcg(L + t);
    L[s] = (b & 0xFFFFFFFF00000000ull) | (unsigned)((unsigned)a + (unsigned)b);
  }
}

// The contour of pixel p in decreasing raster order: (1, points) at an external start, else (0, 0).  *s0 as
// start_state; *k the point count.
__device__ __forceinline__ void contour_of(const Ws& w, const Img& I, long long so, int p, long long* s0, long long* k) {
  int c1;
  *s0 = start_state(I, p, &c1);
  if (*s0 == -1) *k = 0;
  else if (*s0 == -2) *k = 1;
  else {
    const unsigned long long r = w.link[so + *s0];
    const unsigned s1 = (unsigned)r;
    *k = ((w.meta[so + *s0] & KEEP) ? 1 : 0) + (unsigned)w.link[so + s1];
  }
}

// grid (nblk, B): cblk[b][blk] = (contours, points) of the block's pixels, taken in decreasing raster order.
__global__ void __launch_bounds__(PT) ct_count_kernel(Ws w, int H, int W, long long cap, int nblk) {
  const Img I = img(w, blockIdx.y, H, W);
  const long long so = (long long)blockIdx.y * cap;
  const int HW = H * W;
  long long v[2] = {0, 0};
  for (int j = 0; j < PPT; ++j) {
    const int r = blockIdx.x * PB + threadIdx.x * PPT + j;
    if (r >= HW) break;
    long long s0, k;
    contour_of(w, I, so, HW - 1 - r, &s0, &k);
    v[0] += s0 != -1;
    v[1] += k;
  }
  long long e[2], t[2];
  block_scan<2, PT / 32>(v, e, t);
  if (threadIdx.x == 0) {
    long long* o = w.cblk + ((long long)blockIdx.y * nblk + blockIdx.x) * 2;
    o[0] = t[0];
    o[1] = t[1];
  }
}

// grid (nblk, B): offsets_out[coff[b] + k] = contour k's first point (within the image), offsets_out[coff[b] + n_b] =
// N_b; the start points; each root's word becomes (end of its points within the image << 32 | successor), so the call
// can be repeated.
__global__ void __launch_bounds__(PT)
ct_offsets_kernel(Ws w, int H, int W, long long cap, int nblk, const long long* __restrict__ coff,
                  const long long* __restrict__ poff, long long* __restrict__ offsets_out, int2* __restrict__ points_out) {
  const int b = blockIdx.y;
  const Img I = img(w, b, H, W);
  const long long so = (long long)b * cap;
  const int HW = H * W;
  long long s0[PPT], k[PPT], v[2] = {0, 0};
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int r = blockIdx.x * PB + threadIdx.x * PPT + j;
    s0[j] = -1;
    k[j] = 0;
    if (r < HW) contour_of(w, I, so, HW - 1 - r, &s0[j], &k[j]);
    v[0] += s0[j] != -1;
    v[1] += k[j];
  }
  long long e[2], t[2];
  block_scan<2, PT / 32>(v, e, t);
  const long long* cb = w.cblk + ((long long)b * nblk + blockIdx.x) * 2;
  long long ci = cb[0] + e[0], pi = cb[1] + e[1];
  const long long co = coff[b], po = poff[b];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    if (s0[j] == -1) continue;
    const int p = HW - 1 - (blockIdx.x * PB + threadIdx.x * PPT + j);
    offsets_out[co + ci] = pi;
    if (s0[j] == -2 || (w.meta[so + s0[j]] & KEEP)) points_out[po + pi] = make_int2(p % W, p / W);
    if (s0[j] >= 0) w.link[so + s0[j]] = (unsigned long long)(pi + k[j]) << 32 | (unsigned)w.link[so + s0[j]];
    ++ci;
    pi += k[j];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) offsets_out[co + w.ctot[2 * b]] = w.ctot[2 * b + 1];
}

// grid (<= JUMP_MAX_CTAS, B): every kept state that reached a root (other than the root) writes its point.
__global__ void __launch_bounds__(JUMP_T)
ct_points_kernel(int W, long long cap, const long long* __restrict__ stot, const long long* __restrict__ poff,
                 const unsigned* __restrict__ meta, const unsigned long long* __restrict__ link,
                 int2* __restrict__ points_out) {
  const long long so = (long long)blockIdx.y * cap, n = stot[blockIdx.y], po = poff[blockIdx.y];
  const unsigned* M = meta + so;
  const unsigned long long* L = link + so;
  for (long long s = (long long)blockIdx.x * JUMP_T + threadIdx.x; s < n; s += (long long)gridDim.x * JUMP_T) {
    const unsigned m = M[s];
    if ((m & ROOT) || !(m & KEEP)) continue;
    const unsigned long long a = L[s];
    const unsigned t = (unsigned)(a >> 32);
    if (!(M[t] & ROOT)) continue;                    // a hole, a non-external component or a dead chain
    const int p = (int)(m & PIX);
    points_out[po + (long long)(L[t] >> 32) - (unsigned)a] = make_int2(p % W, p / W);
  }
}

int jump_grid(const Layout& L) { return (int)std::min<long long>((L.cap + JUMP_T - 1) / JUMP_T, JUMP_MAX_CTAS); }

}  // namespace

extern "C" size_t rbu_contours_workspace_bytes(int B, int H, int W) {
  if (!dims_ok(B, H, W)) return 0;
  return layout(B, H, W).total;
}

extern "C" int rbu_trace_contours(const void* mask, int kind, float threshold, int B, int H, int W, int approx,
                                  int64_t* counts_out, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(mask && counts_out && workspace, "rbu_trace_contours: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_trace_contours: need 1 <= B <= 65535 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)",
                B, H, W);
  RBU_CHECK_ARG(kind == RBU_KIND_F32 || kind == RBU_KIND_U8, "rbu_trace_contours: kind must be RBU_KIND_F32 or RBU_KIND_U8");
  RBU_CHECK_ARG(approx == RBU_APPROX_NONE || approx == RBU_APPROX_SIMPLE,
                "rbu_trace_contours: approx must be RBU_APPROX_NONE or RBU_APPROX_SIMPLE (got %d)", approx);
  RBU_CHECK_ARG(workspace_bytes >= rbu_contours_workspace_bytes(B, H, W), "rbu_trace_contours: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "rbu_trace_contours: workspace must be 16-byte aligned");
  const Layout L = layout(B, H, W);
  const Ws w = carve(workspace, L);
  const int cx = rbu_cdiv(W, 32), segs = rbu_cdiv((long)H * cx, SEGS);
  int rc = union_find_passes<false, false>(mask, kind, threshold, 0, B, H, W, 1, cx, segs, w.pfg, nullptr, nullptr, stream);
  if (rc != RBU_OK) return rc;
  rc = union_find_passes<false, false>(mask, kind, threshold, 1, B, H, W, 0, cx, segs, w.pbg, nullptr, nullptr, stream);
  if (rc != RBU_OK) return rc;
  ct_frame_kernel<<<dim3(rbu_cdiv(2L * (W + H), 256), B), 256, 0, stream>>>(H, W, w.pbg);
  RBU_CHECK_LAUNCH();
  const dim3 pix(L.nblk, B);
  ct_nb_kernel<<<pix, PT, 0, stream>>>(H, W, L.nblk, w.pfg, w.nb, w.sblk);
  RBU_CHECK_LAUNCH();
  ct_scan_kernel<1><<<B, SCAN_T, 0, stream>>>(L.nblk, w.sblk, w.stot, nullptr);
  RBU_CHECK_LAUNCH();
  ct_base_kernel<<<pix, PT, 0, stream>>>(H * W, L.nblk, w.nb, w.sblk, w.base);
  RBU_CHECK_LAUNCH();
  ct_links_kernel<<<pix, PT, 0, stream>>>(w, H, W, L.cap, approx);
  RBU_CHECK_LAUNCH();
  const dim3 sg(jump_grid(L), B);
  for (int r = 0; r < L.rounds; ++r) {
    ct_jump_kernel<<<sg, JUMP_T, 0, stream>>>(L.cap, w.stot, w.meta, w.link);
    RBU_CHECK_LAUNCH();
  }
  ct_count_kernel<<<pix, PT, 0, stream>>>(w, H, W, L.cap, L.nblk);
  RBU_CHECK_LAUNCH();
  ct_scan_kernel<2><<<B, SCAN_T, 0, stream>>>(L.nblk, w.cblk, w.ctot, reinterpret_cast<long long*>(counts_out));
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}

extern "C" int rbu_write_contours(void* workspace, size_t workspace_bytes, int B, int H, int W,
                                  const int64_t* contour_offsets, const int64_t* point_offsets, int64_t* offsets_out,
                                  int32_t* points_out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RBU_CHECK_ARG(workspace && contour_offsets && point_offsets && offsets_out && points_out,
                "rbu_write_contours: null pointer");
  RBU_CHECK_ARG(dims_ok(B, H, W), "rbu_write_contours: need 1 <= B <= 65535 and 1 <= H, W <= 32768 (got B=%d, H=%d, W=%d)",
                B, H, W);
  RBU_CHECK_ARG(workspace_bytes >= rbu_contours_workspace_bytes(B, H, W), "rbu_write_contours: workspace too small");
  RBU_CHECK_ARG(((uintptr_t)workspace & 15) == 0 && ((uintptr_t)points_out & 7) == 0,
                "rbu_write_contours: workspace must be 16-byte and points_out 8-byte aligned");
  const Layout L = layout(B, H, W);
  const Ws w = carve(workspace, L);
  int2* pts = reinterpret_cast<int2*>(points_out);
  ct_offsets_kernel<<<dim3(L.nblk, B), PT, 0, stream>>>(w, H, W, L.cap, L.nblk,
                                                        reinterpret_cast<const long long*>(contour_offsets),
                                                        reinterpret_cast<const long long*>(point_offsets),
                                                        reinterpret_cast<long long*>(offsets_out), pts);
  RBU_CHECK_LAUNCH();
  ct_points_kernel<<<dim3(jump_grid(L), B), JUMP_T, 0, stream>>>(
      W, L.cap, w.stot, reinterpret_cast<const long long*>(point_offsets), w.meta, w.link, pts);
  RBU_CHECK_LAUNCH();
  return RBU_OK;
}
