// attention.cuh -- fused dot-product graph attention (PyG TransformerConv) over a dst-sorted edge list, sm_100a:
//
//     score[e, h] = scale * < q[dst[e], h, :], k[src[e], h, :] >
//     out[i, h, :] = sum_{e : dst[e] = i} alpha[e, h] * v[src[e], h, :],   alpha = softmax of score over the row i
//     lse[i, h]    = log sum_{e : dst[e] = i} exp(score[e, h])
//
// FlashAttention's online softmax restricted to a graph: one pass keeps a running (m, s, acc[F]) per row and head, so no
// [E, H] score or alpha is stored.  The backward recomputes p = alpha from lse (FlashAttention-2):
//
//     D[i, h] = < g[i, h], out[i, h] >,  p = exp(score - lse[dst]),  dp = < g[dst, h], v[src, h] >,  ds = p (dp - D[dst])
//     grad_q[i] = sum_{e : dst = i} (scale ds) k[src]     (attention_grad_kernel, dst-sorted pass)
//
// and writes p and scale * ds as [E, H]; grad_k and grad_v are mh_spmm passes on the transposed list (mh_spmm.py).
//
//   * Edge-count partition, as gatv2_grad_kernel: a warp owns a CHUNK of `chunk` consecutive edges, a 256-thread CTA a
//     TILE of 8 chunks.  No CTA or warp is assigned per row, so a hub row is spread over many CTAs.
//   * Lane layout: a head is a group of G lanes (a power of two, at most 32), each holding VPH vectors of VECW columns of
//     it; 32 / G heads side by side make a layer, NL layers a launch.  The per-head dot is a butterfly over the low
//     log2(G) lane bits, after which every lane of the group holds the same sum.  A lane holds the q row (re-loaded at
//     each segment head), the running max m and sum s of its head, and its columns of acc.
//   * Online softmax per edge: M = max(m, x), acc = acc exp(m - M) + exp(x - M) v, s likewise.  Two pieces combine as
//     M = max(m1, m2), s = s1 e1 + s2 e2, acc = acc1 e1 + acc2 e2 with ei = exp(mi - M) (0 for mi = -inf).  The max is
//     NaN-propagating, so a NaN score makes its row NaN.
//   * A row inside a chunk is finished by the warp: out = acc / s, lse = m + log s.  A row cut by chunk boundaries
//     leaves a piece in shared memory (s_head: the chunk's first run when the row started earlier; s_tail: its last run
//     when it goes on); after one __syncthreads the chunk where the row starts joins the later pieces left to right.
//     Rows cut by TILE boundaries go through workspace carries: attention_fixup_kernel combines each chain in tile order
//     and writes that row.  Rows without edges get out = 0 and lse = -inf (attention_empty_kernel).
//   * The backward has one carry, the plain sum of grad_q: the same pieces and chains, finished by gatv2_fixup_kernel.
//   * A launch covers whole heads, at most gv_slab() columns; wider rows run as several launches over disjoint heads.
//   * No atomics; the partition depends on E alone, so two calls return the same bits.  bf16 / fp16 / fp32 accumulate
//     in fp32, fp64 in fp64; accurate expf / exp / logf / log, IEEE division, one rounding on every store.
#pragma once
#include "gatv2.cuh"

namespace geot {

// Most accumulator bytes per lane and array: 8 fp32 or 4 fp64 columns, so a warp covers gv_slab() columns.
constexpr int kAttLaneBytes = 32;
template <typename A, int VECW> constexpr int att_kv_max() { return kAttLaneBytes / (VECW * (int)sizeof(A)); }

struct AttentionParams {
  const void *q;                // [N_dst, W], indexed by dst_index (sorted)
  const void *k;                // [N_src, W], indexed by src_index
  const void *v;                // [N_src, W]
  const int64_t *src_index;     // [E]
  const int64_t *dst_index;     // [E], non-decreasing
  void *out;                    // [N_dst, W]: forward output; backward: grad_q
  void *lse;                    // [N_dst, H] accumulator type: forward output; backward input
  const void *o;                // backward: the forward's out [N_dst, W]
  const void *g;                // backward: d loss / d out [N_dst, W]
  void *p_out, *ds_out;         // backward: p and scale * ds [E, H]
  int64_t E, W, H, F;
  int64_t h0;                   // first head of this launch
  int hc;                       // heads of this launch
  int G;                        // lanes per head
  int chunk;                    // edges per warp
  int64_t n_tiles;
  double scale;
  void *carry_head, *carry_tail;   // per tile: forward [wc] acc, [hc] m, [hc] s; backward [wc] acc
  unsigned char *flags;            // [n_tiles] FLAG_HEAD / FLAG_THROUGH / FLAG_TAIL of each tile
};

// Edges whose k and v rows are in flight per warp: 4 while a lane holds at most 16 bytes of accumulators per array,
// else 2.  Shapes of one fp32 vector slot per lane run two CTAs per SM (128 registers); the others, with more slots or
// fp64 accumulators, one CTA with up to 255 registers, so that no shape spills.
template <typename T, int VECW, int KV>
struct AttShape {
  using A = typename AccOf<T>::type;
  static constexpr int acc_bytes = KV * VECW * (int)sizeof(A);
  static constexpr int U = acc_bytes <= 16 ? 4 : 2;
  static constexpr int min_blocks = (KV == 1 && sizeof(A) == 4) ? 2 : 1;
};

template <typename A> __device__ __forceinline__ A att_exp(A x);
template <> __device__ __forceinline__ float att_exp<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ double att_exp<double>(double x) { return exp(x); }
template <typename A> __device__ __forceinline__ A att_log(A x);
template <> __device__ __forceinline__ float att_log<float>(float x) { return logf(x); }
template <> __device__ __forceinline__ double att_log<double>(double x) { return log(x); }

// NaN-propagating max, and the factor exp(m - M) of a piece with max m (0 for an empty piece, m = -inf)
template <typename A> __device__ __forceinline__ A att_max(A a, A b) { return (b > a || b != b) ? b : a; }
template <typename A> __device__ __forceinline__ A att_rescale(A m, A M) { return m == -INFINITY ? A(0) : att_exp(m - M); }

// Sum over the G lanes of each head group (xor butterfly: every lane of the group ends with the same bits).
template <typename A> __device__ __forceinline__ A att_group_sum(A x, int G) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    if (o < G) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// The columns a lane holds: slot (l, j) is vector j of head l * (32 / G) + lane / G of the launch, columns
// [cs, cs + VECW) of the launch's wc = hc * F, where cs = head * F + (j * G + lane % G) * VECW.
template <int NL, int VPH, int VECW>
struct AttLanes {
  int head[NL];            // head of layer l, relative to h0
  bool hv[NL];             // head[l] < hc
  int cs[NL][VPH];         // column of the slot inside the launch
  bool ok[NL][VPH];
  bool lead;               // lane % G == 0: stores the per-head values
  __device__ __forceinline__ AttLanes(int lane, int G, int hc, int64_t F) {
    const int hpl = 32 / G, gi = lane / G, gl = lane % G;
    lead = gl == 0;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      head[l] = l * hpl + gi;
      hv[l] = head[l] < hc;
#pragma unroll
      for (int j = 0; j < VPH; ++j) {
        const int cf = (j * G + gl) * VECW;
        ok[l][j] = hv[l] && cf < F;
        cs[l][j] = ok[l][j] ? head[l] * (int)F + cf : 0;
      }
    }
  }
};

// ---- forward ----------------------------------------------------------------------------------------------------------
template <typename T, int VECW, int NL, int VPH>
__global__ void __launch_bounds__(kThreads, (AttShape<T, VECW, NL * VPH>::min_blocks))
    attention_fwd_kernel(const __grid_constant__ AttentionParams p) {
  using A = typename AccOf<T>::type;
  using VecT = Vec<T, VECW>;
  constexpr int KV = NL * VPH;
  constexpr int U = AttShape<T, VECW, KV>::U;
  extern __shared__ __align__(16) unsigned char att_smem[];
  __shared__ int s_flags[kGvWarps];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hc = p.hc;
  const int wc = hc * (int)p.F;
  const int piece = wc + 2 * hc;                          // [wc] acc, [hc] m, [hc] s
  A *s_head = reinterpret_cast<A *>(att_smem);            // [kGvWarps][piece]
  A *s_tail = s_head + kGvWarps * piece;
  const int64_t E = p.E, W = p.W, H = p.H;
  const int64_t c0 = p.h0 * p.F;
  const int64_t *__restrict__ di = p.dst_index;
  const int64_t *__restrict__ si = p.src_index;
  const T *__restrict__ qb = static_cast<const T *>(p.q) + c0;
  const T *__restrict__ kb = static_cast<const T *>(p.k) + c0;
  const T *__restrict__ vb = static_cast<const T *>(p.v) + c0;
  T *__restrict__ ob = static_cast<T *>(p.out) + c0;
  A *__restrict__ lb = static_cast<A *>(p.lse) + p.h0;
  const A scale = A(p.scale);
  const uint64_t pol = policy_evict_first();

  const int64_t tile = blockIdx.x;
  const int64_t C = p.chunk;
  const int64_t t_begin = tile * kGvWarps * C;
  const int64_t t_end = min(t_begin + kGvWarps * C, E);
  const int64_t first_row = di[t_begin], last_row = di[t_end - 1];
  const bool t_head = t_begin > 0 && di[t_begin - 1] == first_row;
  const bool t_cont = t_end < E && di[t_end] == last_row;
  const int64_t cb = t_begin + warp * C;
  const int64_t ce = min(cb + C, t_end);
  int flags = 0;
  int64_t r1 = 0;
  if (cb < ce) {
    const int64_t r0 = di[cb];
    r1 = di[ce - 1];
    if (cb > 0 && di[cb - 1] == r0) flags |= FLAG_HEAD;
    if (ce < E && di[ce] == r1) flags |= ((flags & FLAG_HEAD) && r0 == r1) ? FLAG_THROUGH : FLAG_TAIL;
  }
  if (lane == 0) s_flags[warp] = flags;

  const AttLanes<NL, VPH, VECW> L(lane, p.G, hc, p.F);
  A qr[NL][VPH][VECW], acc[NL][VPH][VECW], m[NL], s[NL];
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    m[l] = -INFINITY;
    s[l] = A(0);
#pragma unroll
    for (int j = 0; j < VPH; ++j)
#pragma unroll
      for (int i = 0; i < VECW; ++i) qr[l][j][i] = acc[l][j][i] = A(0);
  }
  // a piece: acc by column, then m and s by head (lead lanes)
  auto to_smem = [&](A *dst) {
#pragma unroll
    for (int l = 0; l < NL; ++l) {
#pragma unroll
      for (int j = 0; j < VPH; ++j)
        if (L.ok[l][j])
#pragma unroll
          for (int i = 0; i < VECW; ++i) dst[L.cs[l][j] + i] = acc[l][j][i];
      if (L.hv[l] && L.lead) {
        dst[wc + L.head[l]] = m[l];
        dst[wc + hc + L.head[l]] = s[l];
      }
    }
  };
  auto store_row = [&](int64_t r) {
#pragma unroll
    for (int l = 0; l < NL; ++l) {
#pragma unroll
      for (int j = 0; j < VPH; ++j) {
        if (!L.ok[l][j]) continue;
        VecT o;
#pragma unroll
        for (int i = 0; i < VECW; ++i) o.v[i] = from_acc<T>(acc[l][j][i] / s[l]);
        *reinterpret_cast<VecT *>(ob + r * W + L.cs[l][j]) = o;
      }
      if (L.hv[l] && L.lead) lb[r * H + L.head[l]] = m[l] + att_log(s[l]);
    }
  };

  if (cb < ce) {
    int64_t cur = -1;
    bool first = true;
    for (int64_t b = cb; b < ce; b += 32) {
      const int64_t le = min(b + lane, ce - 1);
      const int64_t my_row = ld_stream(di + le, pol);
      const int64_t my_src = ld_stream(si + le, pol);
      const int n = (int)min((int64_t)32, ce - b);
      for (int k0 = 0; k0 < n; k0 += U) {
        // the k and v rows of U edges leave before the first is used
        VecT kv[U][NL][VPH], vv[U][NL][VPH];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t sr = __shfl_sync(0xffffffffu, my_src, min(k0 + u, n - 1));
#pragma unroll
          for (int l = 0; l < NL; ++l)
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j]) {
                kv[u][l][j] = *reinterpret_cast<const VecT *>(kb + sr * W + L.cs[l][j]);
                vv[u][l][j] = *reinterpret_cast<const VecT *>(vb + sr * W + L.cs[l][j]);
              }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (k0 + u >= n) break;
          const int64_t r = __shfl_sync(0xffffffffu, my_row, k0 + u);
          if (r != cur) {
            if (cur >= 0) {      // the previous run ends inside the chunk
              if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * piece);
              else store_row(cur);
              first = false;
            }
            cur = r;
#pragma unroll
            for (int l = 0; l < NL; ++l) {
              m[l] = -INFINITY;
              s[l] = A(0);
#pragma unroll
              for (int j = 0; j < VPH; ++j) {
                VecT x;
                if (L.ok[l][j]) x = *reinterpret_cast<const VecT *>(qb + r * W + L.cs[l][j]);
#pragma unroll
                for (int i = 0; i < VECW; ++i) {
                  qr[l][j][i] = L.ok[l][j] ? to_acc<T>(x.v[i]) : A(0);
                  acc[l][j][i] = A(0);
                }
              }
            }
          }
#pragma unroll
          for (int l = 0; l < NL; ++l) {
            A d = A(0);
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j])
#pragma unroll
                for (int i = 0; i < VECW; ++i) d += qr[l][j][i] * to_acc<T>(kv[u][l][j].v[i]);
            const A x = scale * att_group_sum(d, p.G);
            const A M = att_max(m[l], x);
            const A e1 = att_rescale(m[l], M);
            const A e2 = att_rescale(x, M);
            m[l] = M;
            s[l] = s[l] * e1 + e2;
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j])
#pragma unroll
                for (int i = 0; i < VECW; ++i) acc[l][j][i] = acc[l][j][i] * e1 + e2 * to_acc<T>(vv[u][l][j].v[i]);
          }
        }
      }
    }
    // the chunk's last run
    if (flags & FLAG_THROUGH) to_smem(s_head + warp * piece);
    else if (flags & FLAG_TAIL) to_smem(s_tail + warp * piece);
    else if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * piece);
    else store_row(cur);
  }
  __syncthreads();

  // ---- chains of pieces inside the tile, left to right ----
  if (cb < ce) {
    auto load_piece = [&](const A *src) {
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        m[l] = L.hv[l] ? src[wc + L.head[l]] : A(0);
        s[l] = L.hv[l] ? src[wc + hc + L.head[l]] : A(0);
#pragma unroll
        for (int j = 0; j < VPH; ++j)
#pragma unroll
          for (int i = 0; i < VECW; ++i) acc[l][j][i] = L.ok[l][j] ? src[L.cs[l][j] + i] : A(0);
      }
    };
    auto add_piece = [&](const A *src) {
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        if (!L.hv[l]) continue;
        const A m2 = src[wc + L.head[l]], s2 = src[wc + hc + L.head[l]];
        const A M = att_max(m[l], m2);
        const A e1 = att_rescale(m[l], M), e2 = att_rescale(m2, M);
        m[l] = M;
        s[l] = s[l] * e1 + s2 * e2;
#pragma unroll
        for (int j = 0; j < VPH; ++j)
          if (L.ok[l][j])
#pragma unroll
            for (int i = 0; i < VECW; ++i) acc[l][j][i] = acc[l][j][i] * e1 + src[L.cs[l][j] + i] * e2;
      }
    };
    auto to_carry = [&](void *carry) { to_smem(static_cast<A *>(carry) + tile * piece); };
    if (warp == 0 && (flags & FLAG_HEAD)) {
      // the row that entered the tile from the left: its tile piece goes to the workspace
      load_piece(s_head);
      for (int j = 0; j + 1 < kGvWarps && (s_flags[j] & FLAG_THROUGH); ++j) add_piece(s_head + (j + 1) * piece);
      to_carry(p.carry_head);
    }
    if (flags & FLAG_TAIL) {
      load_piece(s_tail + warp * piece);
      bool inside = false;
      for (int j = warp + 1; j < kGvWarps; ++j) {
        add_piece(s_head + j * piece);
        if (!(s_flags[j] & FLAG_THROUGH)) { inside = true; break; }
      }
      if (inside) store_row(r1);
      else to_carry(p.carry_tail);      // the row goes on in the next tile
    }
  }
  if (tid == 0) {
    const bool through = t_head && t_cont && first_row == last_row;
    p.flags[tile] = (unsigned char)((t_head ? FLAG_HEAD : 0) | (through ? FLAG_THROUGH : 0) |
                                    ((t_cont && !through) ? FLAG_TAIL : 0));
  }
}

// A chain = tail[t] + head[t+1] + ... + head[last], last the first tile after t that is not THROUGH, combined in that
// order; one warp per chain, lanes over the columns (each lane combines the (m, s) of its column's head alongside) and
// then over the heads for lse.
template <typename T>
__global__ void __launch_bounds__(kThreads) attention_fixup_kernel(const __grid_constant__ AttentionParams p) {
  using A = typename AccOf<T>::type;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (kThreads / 32) + warp;
  if (t >= p.n_tiles || !(p.flags[t] & FLAG_TAIL)) return;
  int64_t last = t + 1;
  for (;;) {   // chain end: scan the THROUGH flags 32 tiles at a time
    const int64_t q = last + lane;
    const bool thr = (q < p.n_tiles) && (p.flags[q] & FLAG_THROUGH);
    const unsigned msk = __ballot_sync(0xffffffffu, !thr);
    if (msk) { last += __ffs(msk) - 1; break; }
    last += 32;
  }
  const int hc = p.hc, F = (int)p.F, wc = hc * F, piece = wc + 2 * hc;
  const int64_t te = kGvWarps * (int64_t)p.chunk;
  const int64_t r = p.dst_index[min((t + 1) * te, p.E) - 1];
  const A *head = static_cast<const A *>(p.carry_head);
  const A *tail = static_cast<const A *>(p.carry_tail);
  // the row's (m, s) of head h, combined in chain order
  auto stats = [&](int h, A &m, A &s) {
    m = tail[t * piece + wc + h];
    s = tail[t * piece + wc + hc + h];
    for (int64_t j = t + 1; j <= last; ++j) {
      const A m2 = head[j * piece + wc + h], s2 = head[j * piece + wc + hc + h];
      const A M = att_max(m, m2);
      s = s * att_rescale(m, M) + s2 * att_rescale(m2, M);
      m = M;
    }
  };
  T *out = static_cast<T *>(p.out) + r * p.W + p.h0 * p.F;
  for (int c = lane; c < wc; c += 32) {
    const int h = c / F;
    A m = tail[t * piece + wc + h], s = tail[t * piece + wc + hc + h], a = tail[t * piece + c];
    for (int64_t j = t + 1; j <= last; ++j) {
      const A m2 = head[j * piece + wc + h], s2 = head[j * piece + wc + hc + h];
      const A M = att_max(m, m2);
      const A e1 = att_rescale(m, M), e2 = att_rescale(m2, M);
      s = s * e1 + s2 * e2;
      a = a * e1 + head[j * piece + c] * e2;
      m = M;
    }
    out[c] = from_acc<T>(a / s);
  }
  A *lse = static_cast<A *>(p.lse) + r * p.H + p.h0;
  for (int h = lane; h < hc; h += 32) {
    A m, s;
    stats(h, m, s);
    lse[h] = m + att_log(s);
  }
}

// Rows of the forward's output that no edge reaches -- beyond the plan's rows, or with rowptr[r] == rowptr[r + 1] --
// get out = 0 and lse = -inf (the log of an empty sum).  One warp per row.
template <typename T>
__global__ void __launch_bounds__(kThreads) attention_empty_kernel(T *out, typename AccOf<T>::type *lse,
                                                                   const int64_t *rowptr, int64_t S_plan, int64_t S_out,
                                                                   int64_t W, int64_t H) {
  using A = typename AccOf<T>::type;
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * kThreads) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5; r < S_out; r += n_warps) {
    if (r < S_plan && rowptr[r] != rowptr[r + 1]) continue;
    for (int64_t c = lane; c < W; c += 32) out[r * W + c] = from_acc<T>(A(0));
    for (int64_t h = lane; h < H; h += 32) lse[r * H + h] = -INFINITY;
  }
}

// out[i] = value, i < n (the all-ones factor that lets gatv2_fixup_kernel finish grad_q).
template <typename T>
__global__ void __launch_bounds__(kThreads) attention_fill_kernel(T *out, int64_t n, float value) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads)
    out[i] = from_acc<T>(typename AccOf<T>::type(value));
}

// ---- backward, dst pass -----------------------------------------------------------------------------------------------
template <typename T, int VECW, int NL, int VPH>
__global__ void __launch_bounds__(kThreads, (AttShape<T, VECW, NL * VPH>::min_blocks))
    attention_grad_kernel(const __grid_constant__ AttentionParams p) {
  using A = typename AccOf<T>::type;
  using VecT = Vec<T, VECW>;
  constexpr int KV = NL * VPH;
  constexpr int U = AttShape<T, VECW, KV>::U;
  extern __shared__ __align__(16) unsigned char att_smem[];
  __shared__ int s_flags[kGvWarps];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hc = p.hc;
  const int wc = hc * (int)p.F;
  A *s_head = reinterpret_cast<A *>(att_smem);            // [kGvWarps][wc]
  A *s_tail = s_head + kGvWarps * wc;
  const int64_t E = p.E, W = p.W, H = p.H;
  const int64_t c0 = p.h0 * p.F;
  const int64_t *__restrict__ di = p.dst_index;
  const int64_t *__restrict__ si = p.src_index;
  const T *__restrict__ qb = static_cast<const T *>(p.q) + c0;
  const T *__restrict__ kb = static_cast<const T *>(p.k) + c0;
  const T *__restrict__ vb = static_cast<const T *>(p.v) + c0;
  const T *__restrict__ obase = static_cast<const T *>(p.o) + c0;
  const T *__restrict__ gb = static_cast<const T *>(p.g) + c0;
  const A *__restrict__ lb = static_cast<const A *>(p.lse) + p.h0;
  T *__restrict__ gq = static_cast<T *>(p.out) + c0;
  T *__restrict__ pw = static_cast<T *>(p.p_out) + p.h0;
  T *__restrict__ dw = static_cast<T *>(p.ds_out) + p.h0;
  const A scale = A(p.scale);
  const uint64_t pol = policy_evict_first();

  const int64_t tile = blockIdx.x;
  const int64_t C = p.chunk;
  const int64_t t_begin = tile * kGvWarps * C;
  const int64_t t_end = min(t_begin + kGvWarps * C, E);
  const int64_t first_row = di[t_begin], last_row = di[t_end - 1];
  const bool t_head = t_begin > 0 && di[t_begin - 1] == first_row;
  const bool t_cont = t_end < E && di[t_end] == last_row;
  const int64_t cb = t_begin + warp * C;
  const int64_t ce = min(cb + C, t_end);
  int flags = 0;
  int64_t r1 = 0;
  if (cb < ce) {
    const int64_t r0 = di[cb];
    r1 = di[ce - 1];
    if (cb > 0 && di[cb - 1] == r0) flags |= FLAG_HEAD;
    if (ce < E && di[ce] == r1) flags |= ((flags & FLAG_HEAD) && r0 == r1) ? FLAG_THROUGH : FLAG_TAIL;
  }
  if (lane == 0) s_flags[warp] = flags;

  const AttLanes<NL, VPH, VECW> L(lane, p.G, hc, p.F);
  A qr[NL][VPH][VECW], gr[NL][VPH][VECW], acc[NL][VPH][VECW], D[NL], lse[NL];
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    D[l] = lse[l] = A(0);
#pragma unroll
    for (int j = 0; j < VPH; ++j)
#pragma unroll
      for (int i = 0; i < VECW; ++i) qr[l][j][i] = gr[l][j][i] = acc[l][j][i] = A(0);
  }
  auto to_smem = [&](A *dst) {
#pragma unroll
    for (int l = 0; l < NL; ++l)
#pragma unroll
      for (int j = 0; j < VPH; ++j)
        if (L.ok[l][j])
#pragma unroll
          for (int i = 0; i < VECW; ++i) dst[L.cs[l][j] + i] = acc[l][j][i];
  };
  auto store_row = [&](int64_t r) {
#pragma unroll
    for (int l = 0; l < NL; ++l)
#pragma unroll
      for (int j = 0; j < VPH; ++j) {
        if (!L.ok[l][j]) continue;
        VecT o;
#pragma unroll
        for (int i = 0; i < VECW; ++i) o.v[i] = from_acc<T>(acc[l][j][i]);
        *reinterpret_cast<VecT *>(gq + r * W + L.cs[l][j]) = o;
      }
  };

  if (cb < ce) {
    int64_t cur = -1;
    bool first = true;
    for (int64_t b = cb; b < ce; b += 32) {
      const int64_t le = min(b + lane, ce - 1);
      const int64_t my_row = ld_stream(di + le, pol);
      const int64_t my_src = ld_stream(si + le, pol);
      const int n = (int)min((int64_t)32, ce - b);
      for (int k0 = 0; k0 < n; k0 += U) {
        VecT kv[U][NL][VPH], vv[U][NL][VPH];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t sr = __shfl_sync(0xffffffffu, my_src, min(k0 + u, n - 1));
#pragma unroll
          for (int l = 0; l < NL; ++l)
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j]) {
                kv[u][l][j] = *reinterpret_cast<const VecT *>(kb + sr * W + L.cs[l][j]);
                vv[u][l][j] = *reinterpret_cast<const VecT *>(vb + sr * W + L.cs[l][j]);
              }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (k0 + u >= n) break;
          const int64_t r = __shfl_sync(0xffffffffu, my_row, k0 + u);
          if (r != cur) {
            if (cur >= 0) {
              if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * wc);
              else store_row(cur);
              first = false;
            }
            cur = r;
            // the row's q and g in registers, D = <g, out> and lse per head
#pragma unroll
            for (int l = 0; l < NL; ++l) {
              A d = A(0);
#pragma unroll
              for (int j = 0; j < VPH; ++j) {
                VecT xq, xg, xo;
                if (L.ok[l][j]) {
                  xq = *reinterpret_cast<const VecT *>(qb + r * W + L.cs[l][j]);
                  xg = *reinterpret_cast<const VecT *>(gb + r * W + L.cs[l][j]);
                  xo = *reinterpret_cast<const VecT *>(obase + r * W + L.cs[l][j]);
                }
#pragma unroll
                for (int i = 0; i < VECW; ++i) {
                  qr[l][j][i] = L.ok[l][j] ? to_acc<T>(xq.v[i]) : A(0);
                  gr[l][j][i] = L.ok[l][j] ? to_acc<T>(xg.v[i]) : A(0);
                  if (L.ok[l][j]) d += gr[l][j][i] * to_acc<T>(xo.v[i]);
                  acc[l][j][i] = A(0);
                }
              }
              D[l] = att_group_sum(d, p.G);
              lse[l] = L.hv[l] ? lb[r * H + L.head[l]] : A(0);
            }
          }
          const int64_t e = b + k0 + u;
#pragma unroll
          for (int l = 0; l < NL; ++l) {
            A dq = A(0), dv = A(0);
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j])
#pragma unroll
                for (int i = 0; i < VECW; ++i) {
                  dq += qr[l][j][i] * to_acc<T>(kv[u][l][j].v[i]);
                  dv += gr[l][j][i] * to_acc<T>(vv[u][l][j].v[i]);
                }
            const A x = scale * att_group_sum(dq, p.G);
            const A pe = att_exp(x - lse[l]);
            const A sds = scale * (pe * (att_group_sum(dv, p.G) - D[l]));
            if (L.hv[l] && L.lead) {
              pw[e * H + L.head[l]] = from_acc<T>(pe);
              dw[e * H + L.head[l]] = from_acc<T>(sds);
            }
#pragma unroll
            for (int j = 0; j < VPH; ++j)
              if (L.ok[l][j])
#pragma unroll
                for (int i = 0; i < VECW; ++i) acc[l][j][i] += sds * to_acc<T>(kv[u][l][j].v[i]);
          }
        }
      }
    }
    if (flags & FLAG_THROUGH) to_smem(s_head + warp * wc);
    else if (flags & FLAG_TAIL) to_smem(s_tail + warp * wc);
    else if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * wc);
    else store_row(cur);
  }
  __syncthreads();

  // ---- chains of pieces inside the tile, left to right (plain sums) ----
  if (cb < ce) {
    auto load_piece = [&](const A *src) {
#pragma unroll
      for (int l = 0; l < NL; ++l)
#pragma unroll
        for (int j = 0; j < VPH; ++j)
#pragma unroll
          for (int i = 0; i < VECW; ++i) acc[l][j][i] = L.ok[l][j] ? src[L.cs[l][j] + i] : A(0);
    };
    auto add_piece = [&](const A *src) {
#pragma unroll
      for (int l = 0; l < NL; ++l)
#pragma unroll
        for (int j = 0; j < VPH; ++j)
          if (L.ok[l][j])
#pragma unroll
            for (int i = 0; i < VECW; ++i) acc[l][j][i] += src[L.cs[l][j] + i];
    };
    auto to_carry = [&](void *carry) { to_smem(static_cast<A *>(carry) + tile * wc); };
    if (warp == 0 && (flags & FLAG_HEAD)) {
      load_piece(s_head);
      for (int j = 0; j + 1 < kGvWarps && (s_flags[j] & FLAG_THROUGH); ++j) add_piece(s_head + (j + 1) * wc);
      to_carry(p.carry_head);
    }
    if (flags & FLAG_TAIL) {
      load_piece(s_tail + warp * wc);
      bool inside = false;
      for (int j = warp + 1; j < kGvWarps; ++j) {
        add_piece(s_head + j * wc);
        if (!(s_flags[j] & FLAG_THROUGH)) { inside = true; break; }
      }
      if (inside) store_row(r1);
      else to_carry(p.carry_tail);
    }
  }
  if (tid == 0) {
    const bool through = t_head && t_cont && first_row == last_row;
    p.flags[tile] = (unsigned char)((t_head ? FLAG_HEAD : 0) | (through ? FLAG_THROUGH : 0) |
                                    ((t_cont && !through) ? FLAG_TAIL : 0));
  }
}

}  // namespace geot
