// softmax.cuh -- segment softmax over a dst-sorted edge list, and its backward, on sm_100a.
//
//   forward   out[e, h] = exp(src[e, h] - m[r, h]) / sum_{e' in r} exp(src[e', h] - m[r, h]),  m[r, h] = max_{e' in r} src[e', h]
//   backward  grad_src[e, h] = out[e, h] * (grad_out[e, h] - sum_{e' in r} out[e', h] * grad_out[e', h])
// over the edges e of dst row r = dst_index[e]; src / out / grad are [E, H] row-major.
//
//   * Edge-count partition, as segment_reduce_kernel: a thread owns a CHUNK of kSmChunk consecutive edges for one head,
//     a 256-thread CTA owns a TILE of nc = 256 / hp chunks (hp = min(H, 256) heads side by side, so the hp threads of a
//     chunk read one edge's heads as one contiguous piece).  Every CTA does the same work whatever the degree skew.
//   * The carry of a row piece is (max, sum of exp(x - max)) forward, (sum of out * grad) backward.  Two forward pieces
//     combine as M = max(m1, m2), s = s1 exp(m1 - M) + s2 exp(m2 - M); a piece whose max is -inf adds nothing.
//   * Pass 1 computes the pieces of the rows cut by chunk boundaries (a chunk's first and last run) into shared memory;
//     the owner of a chain of pieces (the chunk where the row starts) combines them left to right.  Rows cut by a TILE
//     boundary leave the CTA: their tile pieces go to the workspace, segment_softmax_fixup_kernel combines each chain
//     (32 lanes striding over it, then a fixed tree) into the row's final statistics, and segment_softmax_finish_kernel
//     writes the outputs of those rows.  Pass 2 writes every row that lies inside the tile.
//   * No atomics; the combine order depends on (E, H) alone, so two calls return the same bits.  fp32 / bf16 / fp16
//     accumulate in fp32, fp64 in fp64; accurate exp (expf / exp), IEEE division, one rounding on the store.
#pragma once
#include "segment_reduce.cuh"

namespace geot {

constexpr int kSmChunk = 8;   // edges per thread chunk

struct SoftmaxParams {
  const void *x;               // forward: src logits; backward: out
  const void *g;               // backward: grad_out (forward: null)
  const int64_t *dst_index;
  void *y;                     // forward: out; backward: grad_src
  int64_t E;
  int H;
  int hp;                      // heads per pass: min(H, kThreads)
  int nc;                      // chunks per tile: kThreads / hp
  int64_t n_tiles;
  void *carry_head, *carry_tail;   // [n_tiles][H] SmPair: the pieces of the rows cut by tile boundaries
  void *stat_head, *stat_tail;     // [n_tiles][H] SmPair: their final statistics (fixup kernel)
  unsigned char *flags;            // [n_tiles] FLAG_HEAD / FLAG_THROUGH / FLAG_TAIL of each tile
};

// forward: (m, s) = (max, sum of exp(x - max)); backward: m = sum of out * grad, s unused
template <typename A> struct SmPair { A m, s; };

__device__ __forceinline__ float sm_exp(float v) { return expf(v); }
__device__ __forceinline__ double sm_exp(double v) { return exp(v); }

template <typename A, bool BWD> __device__ __forceinline__ SmPair<A> sm_identity() {
  if constexpr (BWD) return {A(0), A(0)};
  else return {-INFINITY, A(0)};
}

// pieces combine in a fixed order: p is the left one
template <typename A, bool BWD> __device__ __forceinline__ SmPair<A> sm_combine(SmPair<A> p, SmPair<A> q) {
  if constexpr (BWD) return {p.m + q.m, A(0)};
  const A M = (q.m > p.m || q.m != q.m) ? q.m : p.m;       // NaN-propagating max
  const A a = p.m == -INFINITY ? A(0) : p.s * sm_exp(p.m - M);
  const A b = q.m == -INFINITY ? A(0) : q.s * sm_exp(q.m - M);
  return {M, a + b};
}

template <typename T, bool BWD> __device__ __forceinline__ void sm_add(SmPair<typename AccOf<T>::type> &p, const T *x,
                                                                     const T *g, int64_t i) {
  using A = typename AccOf<T>::type;
  const A v = to_acc<T>(__ldg(x + i));
  if constexpr (BWD) {
    p.m += v * to_acc<T>(__ldg(g + i));
  } else if (v <= p.m) {
    if (v != -INFINITY) p.s += sm_exp(v - p.m);             // (+inf twice: exp(inf - inf) = NaN, as torch.softmax)
  } else if (v > p.m) {
    p.s = p.s * sm_exp(p.m - v) + sm_exp(v - v);           // exp(v - v): 1, or NaN for v = +inf
    p.m = v;
  } else {                                                  // a NaN, now or before: the row is NaN
    p.m = p.m + v;
    p.s = p.m;
  }
}

template <typename T, bool BWD> __device__ __forceinline__ void sm_store(const SoftmaxParams &p, int64_t i,
                                                                       SmPair<typename AccOf<T>::type> st) {
  using A = typename AccOf<T>::type;
  const A v = to_acc<T>(__ldg(static_cast<const T *>(p.x) + i));
  A r;
  if constexpr (BWD) r = v * (to_acc<T>(__ldg(static_cast<const T *>(p.g) + i)) - st.m);
  else r = sm_exp(v - st.m) / st.s;
  static_cast<T *>(p.y)[i] = from_acc<T>(r);
}

template <typename T, bool BWD>
__global__ void __launch_bounds__(kThreads, 2) segment_softmax_kernel(const __grid_constant__ SoftmaxParams p) {
  using A = typename AccOf<T>::type;
  using P = SmPair<A>;
  // per (chunk, head) slot c * hp + hl: the chunk's first-run piece, last-run piece, and the final statistics of both
  __shared__ P s_head[kThreads], s_tail[kThreads], s_fin_head[kThreads], s_fin_tail[kThreads];
  __shared__ int s_flags[kThreads];   // per chunk

  const int tid = threadIdx.x;
  const int hp = p.hp, nc = p.nc, H = p.H;
  const int c = tid / hp, hl = tid % hp;
  const bool active = c < nc;
  const int64_t E = p.E;
  const int64_t *__restrict__ di = p.dst_index;
  const T *x = static_cast<const T *>(p.x);
  const T *g = static_cast<const T *>(p.g);
  const int64_t tile = blockIdx.x;
  const int64_t t_begin = tile * nc * (int64_t)kSmChunk;
  const int64_t t_end = min(t_begin + nc * (int64_t)kSmChunk, E);
  const int64_t first_row = di[t_begin], last_row = di[t_end - 1];
  const bool t_head = t_begin > 0 && di[t_begin - 1] == first_row;   // the tile's first row started in an earlier tile
  const bool t_cont = t_end < E && di[t_end] == last_row;            // ... its last row goes on in a later tile

  const int64_t cb = t_begin + (int64_t)c * kSmChunk;
  const int64_t ce = min(cb + kSmChunk, t_end);
  int flags = 0;
  int64_t r0 = 0, r1 = 0;
  if (active && cb < ce) {
    r0 = di[cb];
    r1 = di[ce - 1];
    if (cb > 0 && di[cb - 1] == r0) flags |= FLAG_HEAD;
    if (ce < E && di[ce] == r1) flags |= ((flags & FLAG_HEAD) && r0 == r1) ? FLAG_THROUGH : FLAG_TAIL;
  }
  if (active && hl == 0) s_flags[c] = flags;

  for (int h0 = 0; h0 < H; h0 += hp) {
    const int h = h0 + hl;
    const bool mine = active && cb < ce && h < H;
    // ---- pass 1: the pieces of the runs cut by chunk boundaries ----
    if (mine) {
      if (flags & FLAG_HEAD) {
        P a = sm_identity<A, BWD>();
        for (int64_t e = cb; e < ce && di[e] == r0; ++e) sm_add<T, BWD>(a, x, g, e * H + h);
        s_head[tid] = a;
      }
      if (flags & FLAG_TAIL) {
        int64_t e = ce - 1;
        while (e > cb && di[e - 1] == r1) --e;
        P a = sm_identity<A, BWD>();
        for (; e < ce; ++e) sm_add<T, BWD>(a, x, g, e * H + h);
        s_tail[tid] = a;
      }
    }
    __syncthreads();
    // ---- chains inside the tile, left to right ----
    if (mine) {
      if (c == 0 && (flags & FLAG_HEAD)) {
        // the row that entered the tile from the left: its tile piece goes to the workspace
        P a = s_head[hl];
        for (int j = 0; j + 1 < nc && (s_flags[j] & FLAG_THROUGH); ++j) a = sm_combine<A, BWD>(a, s_head[(j + 1) * hp + hl]);
        static_cast<P *>(p.carry_head)[tile * H + h] = a;
      }
      if (flags & FLAG_TAIL) {
        P a = s_tail[tid];
        int j = c + 1;
        bool inside = false;
        for (; j < nc; ++j) {
          a = sm_combine<A, BWD>(a, s_head[j * hp + hl]);
          if (!(s_flags[j] & FLAG_THROUGH)) { inside = true; break; }
        }
        if (inside) {
          s_fin_tail[tid] = a;
          for (int k = c + 1; k <= j; ++k) s_fin_head[k * hp + hl] = a;
        } else {
          static_cast<P *>(p.carry_tail)[tile * H + h] = a;   // the row goes on in the next tile
        }
      }
    }
    __syncthreads();
    // ---- pass 2: the outputs of the rows inside the tile ----
    if (mine) {
      int64_t e = cb;
      while (e < ce) {
        const int64_t r = di[e];
        int64_t e2 = e + 1;
        while (e2 < ce && di[e2] == r) ++e2;
        const bool deferred = (t_head && r == first_row) || (t_cont && r == last_row);   // finish kernel
        if (!deferred) {
          P st;
          if (e == cb && (flags & FLAG_HEAD)) st = s_fin_head[tid];
          else if (e2 == ce && (flags & FLAG_TAIL)) st = s_fin_tail[tid];
          else {
            st = sm_identity<A, BWD>();
            for (int64_t k = e; k < e2; ++k) sm_add<T, BWD>(st, x, g, k * H + h);
          }
          for (int64_t k = e; k < e2; ++k) sm_store<T, BWD>(p, k * H + h, st);
        }
        e = e2;
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    const bool through = t_head && t_cont && first_row == last_row;
    p.flags[tile] = (unsigned char)((t_head ? FLAG_HEAD : 0) | (through ? FLAG_THROUGH : 0) |
                                    ((t_cont && !through) ? FLAG_TAIL : 0));
  }
}

// A chain = tail[t] + head[t+1] + ... + head[last], last the first tile after t that is not THROUGH.  One warp per
// chain: lane l combines head[t+1+l], head[t+1+l+32], ... in order, a fixed tree brings the 32 partials to lane 0,
// and the tail piece goes in front.  The statistics go to every tile of the chain.
template <typename T, bool BWD>
__global__ void __launch_bounds__(kThreads) segment_softmax_fixup_kernel(const __grid_constant__ SoftmaxParams p) {
  using A = typename AccOf<T>::type;
  using P = SmPair<A>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (kThreads / 32) + warp;
  if (t >= p.n_tiles || !(p.flags[t] & FLAG_TAIL)) return;
  int64_t last = t + 1;
  for (;;) {   // chain end: scan the THROUGH flags 32 tiles at a time
    const int64_t q = last + lane;
    const bool thr = (q < p.n_tiles) && (p.flags[q] & FLAG_THROUGH);
    const unsigned m = __ballot_sync(0xffffffffu, !thr);
    if (m) { last += __ffs(m) - 1; break; }
    last += 32;
  }
  const int H = p.H;
  const P *head = static_cast<const P *>(p.carry_head);
  for (int h = 0; h < H; ++h) {
    P a = sm_identity<A, BWD>();
    for (int64_t j = t + 1 + lane; j <= last; j += 32) a = sm_combine<A, BWD>(a, head[j * H + h]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      P b;
      b.m = __shfl_down_sync(0xffffffffu, a.m, o);
      b.s = __shfl_down_sync(0xffffffffu, a.s, o);
      a = sm_combine<A, BWD>(a, b);   // lanes >= 32 - o combine garbage that never reaches lane 0
    }
    a = sm_combine<A, BWD>(static_cast<const P *>(p.carry_tail)[t * H + h], a);
    a.m = __shfl_sync(0xffffffffu, a.m, 0);
    a.s = __shfl_sync(0xffffffffu, a.s, 0);
    if (lane == 0) static_cast<P *>(p.stat_tail)[t * H + h] = a;
    for (int64_t j = t + 1 + lane; j <= last; j += 32) static_cast<P *>(p.stat_head)[j * H + h] = a;
  }
}

// The outputs of the rows cut by tile boundaries: the tile's first row (when it started in an earlier tile) and its
// last row (when it goes on in a later one), from the statistics of the fixup kernel.
template <typename T, bool BWD>
__global__ void __launch_bounds__(kThreads) segment_softmax_finish_kernel(const __grid_constant__ SoftmaxParams p) {
  using A = typename AccOf<T>::type;
  using P = SmPair<A>;
  const int64_t tile = blockIdx.x;
  const int f = p.flags[tile];
  if (!f) return;
  const int64_t *__restrict__ di = p.dst_index;
  const int64_t t_begin = tile * p.nc * (int64_t)kSmChunk;
  const int64_t t_end = min(t_begin + p.nc * (int64_t)kSmChunk, p.E);
  const int H = p.H;
  // [t_begin, he): the first row (HEAD / THROUGH); [ts, t_end): the last row (TAIL); binary searches in the sorted index
  int64_t he = t_begin, ts = t_end;
  if (f & (FLAG_HEAD | FLAG_THROUGH)) {
    const int64_t r = di[t_begin];
    int64_t lo = t_begin, hi = t_end;   // first edge with a larger row
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (di[mid] <= r) lo = mid + 1; else hi = mid; }
    he = lo;
  }
  if (f & FLAG_TAIL) {
    const int64_t r = di[t_end - 1];
    int64_t lo = t_begin, hi = t_end;   // first edge of the last row
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (di[mid] < r) lo = mid + 1; else hi = mid; }
    ts = lo;
  }
  // (a tile holds at most max(2048, 8 H) elements: 32-bit offsets)
  const unsigned n_head = (unsigned)((he - t_begin) * H), n_tail = (unsigned)((t_end - ts) * H), uH = (unsigned)H;
  for (unsigned i = threadIdx.x; i < n_head; i += kThreads)
    sm_store<T, BWD>(p, t_begin * H + i, static_cast<const P *>(p.stat_head)[tile * H + i % uH]);
  for (unsigned i = threadIdx.x; i < n_tail; i += kThreads)
    sm_store<T, BWD>(p, ts * H + i, static_cast<const P *>(p.stat_tail)[tile * H + i % uH]);
}

}  // namespace geot
