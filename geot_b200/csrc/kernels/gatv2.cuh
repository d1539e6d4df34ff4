// gatv2.cuh -- backward of the GATv2 attention score on sm_100a.  The forward,
//
//     score[e, h] = sum_f att[h, f] * leaky_relu(x_l[src[e], h, f] + x_r[dst[e], h, f])
//
// is the SDDMM launcher with the GATv2 elementwise step (sddmm.cuh, OP = SDDMM_GATV2).  Its gradients are segment
// sums of a per-edge message.  With u = x_row[row[e]] + x_gat[gat[e]] and g = d loss / d score:
//
//     grad_row[r, c] = att[c] * sum_{e : row[e] = r} g[e, c / F] * leaky'(u[e, c])        leaky'(u) = u > 0 ? 1 : slope
//     grad_att[c]    =          sum_e               g[e, c / F] * leaky(u[e, c])
//
// u is symmetric in its two operands, so one kernel serves both node gradients: the dst pass runs over the dst-sorted
// edge list (row = x_r, gathered = x_l) and also produces grad_att; the src pass runs over the transposed, src-sorted
// list (row = x_l, gathered = x_r).  The row sum is column by column, so a row wider than a warp holds is run as
// column slabs of at most gv_slab() columns, one launch each.
//
//   * Edge-count partition, as segment_reduce_kernel: a warp owns a CHUNK of `chunk` consecutive edges, a 256-thread
//     CTA a TILE of 8 chunks.  A lane holds KV vectors of VECW columns of the row in registers: the x_row row (re-loaded
//     at each segment head), the row's accumulator and its share of the grad_att partial.
//     The gathered rows of U edges are in flight at once.
//   * att is factored out of the row sum: the carries are plain sums and att multiplies once, at the store.
//   * A row that lies inside a chunk is stored directly.  A row cut by chunk boundaries leaves a piece in shared memory
//     (s_head: the chunk's first run when the row started earlier; s_tail: its last run when the row goes on); after one
//     __syncthreads the chunk where the row starts adds the later pieces left to right.  Rows cut by TILE boundaries go
//     through workspace carries; gatv2_fixup_kernel adds each chain in tile order.  Rows without edges are zeroed by
//     gatv2_zero_kernel from the plan's row pointers.
//   * grad_att: the 8 warp partials of a tile are added in warp order into one [W] partial per tile (workspace);
//     gatv2_att_kernel adds those in a fixed order (two levels) and rounds once.
//   * No atomics; the partition depends on E alone, so two calls return the same bits.  bf16 / fp16 / fp32 accumulate
//     in fp32, fp64 in fp64; one rounding on every store.
#pragma once
#include "sddmm.cuh"

namespace geot {

constexpr int kGvWarps = kThreads / 32;   // chunks per tile
constexpr int kGvAttSlices = 256;         // first-level slices of the grad_att sum

// Most columns of one launch: 256 for fp32 accumulators, 128 for fp64 (24 KB of shared memory per CTA either way).
template <typename A> constexpr int gv_slab() { return sizeof(A) == 8 ? 128 : 256; }

struct Gatv2GradParams {
  const void *x_row;            // [N_row, W], indexed by row_index (sorted)
  const void *x_gat;            // [N_gat, W], indexed by gat_index
  const void *att;              // [W]
  const void *grad;             // [E, H]: d loss / d score in this pass's edge order
  const int64_t *row_index;     // [E]
  const int64_t *gat_index;     // [E]
  void *grad_row;               // [S_out, W]
  int64_t E, W, H, F;
  int64_t c0;                   // first column of this launch's slab
  int wc;                       // columns of the slab
  int chunk;                    // edges per warp
  int64_t n_tiles;
  double slope;
  void *carry_head, *carry_tail;   // [n_tiles][wc] accumulator: the tile pieces of the rows cut by tile boundaries
  void *att_part;                  // [n_tiles][wc] accumulator: grad_att partial per tile; null: not requested
  unsigned char *flags;            // [n_tiles] FLAG_HEAD / FLAG_THROUGH / FLAG_TAIL of each tile
};

// Gathered rows in flight per warp: 8 while a lane holds one vector of at most 16 bytes of accumulators, else 4, and 2
// for the element-wise shapes of 8 columns per lane.  Those (rows of 129 - 256 element-wise columns) run one CTA per SM
// with up to 255 registers; every other shape two.  (No shape spills: profiles/r03c_gatv2_resource_usage.md.)
template <typename T, int VECW, int KV>
struct GvShape {
  using A = typename AccOf<T>::type;
  static constexpr int acc_bytes = KV * VECW * (int)sizeof(A);   // per lane and accumulator array
  static constexpr int U = (KV == 1 && acc_bytes <= 16) ? 8 : acc_bytes <= 16 ? 4 : (VECW == 1 && KV >= 8) ? 2 : 4;
  static constexpr int min_blocks = (VECW == 1 && KV >= 4) ? 1 : 2;
};

template <typename T, int VECW, int KV>
__global__ void __launch_bounds__(kThreads, (GvShape<T, VECW, KV>::min_blocks))
    gatv2_grad_kernel(const __grid_constant__ Gatv2GradParams p) {
  using A = typename AccOf<T>::type;
  using VecT = Vec<T, VECW>;
  constexpr int U = GvShape<T, VECW, KV>::U;
  extern __shared__ __align__(16) unsigned char gv_smem[];
  __shared__ int s_flags[kGvWarps];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wc = p.wc;
  A *s_head = reinterpret_cast<A *>(gv_smem);            // [kGvWarps][wc]
  A *s_tail = s_head + kGvWarps * wc;
  A *s_att = s_tail + kGvWarps * wc;
  const int64_t E = p.E, W = p.W, H = p.H;
  const int64_t *__restrict__ ri = p.row_index;
  const int64_t *__restrict__ gi = p.gat_index;
  const T *__restrict__ xr_base = static_cast<const T *>(p.x_row) + p.c0;
  const T *__restrict__ xg_base = static_cast<const T *>(p.x_gat) + p.c0;
  const T *__restrict__ grad = static_cast<const T *>(p.grad);
  T *__restrict__ out = static_cast<T *>(p.grad_row) + p.c0;
  const A slope = A(p.slope);
  const uint64_t pol = policy_evict_first();

  const int64_t tile = blockIdx.x;
  const int64_t C = p.chunk;
  const int64_t t_begin = tile * kGvWarps * C;
  const int64_t t_end = min(t_begin + kGvWarps * C, E);
  const int64_t first_row = ri[t_begin], last_row = ri[t_end - 1];
  const bool t_head = t_begin > 0 && ri[t_begin - 1] == first_row;   // the tile's first row started in an earlier tile
  const bool t_cont = t_end < E && ri[t_end] == last_row;            // ... its last row goes on in a later tile
  const int64_t cb = t_begin + warp * C;
  const int64_t ce = min(cb + C, t_end);
  int flags = 0;
  int64_t r1 = 0;
  if (cb < ce) {
    const int64_t r0 = ri[cb];
    r1 = ri[ce - 1];
    if (cb > 0 && ri[cb - 1] == r0) flags |= FLAG_HEAD;
    if (ce < E && ri[ce] == r1) flags |= ((flags & FLAG_HEAD) && r0 == r1) ? FLAG_THROUGH : FLAG_TAIL;
  }
  if (lane == 0) s_flags[warp] = flags;

  // This lane's columns of the slab: vector k covers [lc[k], lc[k] + VECW), inside one head (F % VECW == 0).  att is
  // read at the stores only (a row's sum is multiplied once), so it takes no registers in the edge loop.
  const T *__restrict__ att = static_cast<const T *>(p.att) + p.c0;
  int lc[KV];
  bool ok[KV];
  int64_t head[KV];
  A xr[KV][VECW], acc[KV][VECW], aacc[KV][VECW];
#pragma unroll
  for (int k = 0; k < KV; ++k) {
    lc[k] = (k * 32 + lane) * VECW;
    ok[k] = lc[k] < wc;
    head[k] = ok[k] ? (p.c0 + lc[k]) / p.F : 0;
#pragma unroll
    for (int i = 0; i < VECW; ++i) xr[k][i] = acc[k][i] = aacc[k][i] = A(0);
  }
  auto to_smem = [&](A *dst) {
#pragma unroll
    for (int k = 0; k < KV; ++k)
      if (ok[k])
#pragma unroll
        for (int i = 0; i < VECW; ++i) dst[lc[k] + i] = acc[k][i];
  };
  auto store_row = [&](int64_t r, const A (&s)[KV][VECW]) {
#pragma unroll
    for (int k = 0; k < KV; ++k) {
      if (!ok[k]) continue;
      const VecT w = *reinterpret_cast<const VecT *>(att + lc[k]);
      VecT v;
#pragma unroll
      for (int i = 0; i < VECW; ++i) v.v[i] = from_acc<T>(to_acc<T>(w.v[i]) * s[k][i]);
      *reinterpret_cast<VecT *>(out + r * W + lc[k]) = v;
    }
  };

  if (cb < ce) {
    int64_t cur = -1;
    bool first = true;
    for (int64_t b = cb; b < ce; b += 32) {
      const int64_t le = min(b + lane, ce - 1);
      const int64_t my_row = ld_stream(ri + le, pol);
      const int64_t my_gat = ld_stream(gi + le, pol);
      const int n = (int)min((int64_t)32, ce - b);
      for (int k0 = 0; k0 < n; k0 += U) {
        // the gathered rows and grad values of U edges leave before the first is used
        VecT v[U][KV];
        A gv[U][KV];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t gr = __shfl_sync(0xffffffffu, my_gat, min(k0 + u, n - 1));
          const int64_t e = b + min(k0 + u, n - 1);
#pragma unroll
          for (int k = 0; k < KV; ++k) {
            if (ok[k]) {
              v[u][k] = *reinterpret_cast<const VecT *>(xg_base + gr * W + lc[k]);
              gv[u][k] = to_acc<T>(__ldg(grad + e * H + head[k]));
            }
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (k0 + u >= n) break;
          const int64_t r = __shfl_sync(0xffffffffu, my_row, k0 + u);
          if (r != cur) {
            if (cur >= 0) {      // the previous run ends inside the chunk
              if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * wc);
              else store_row(cur, acc);
              first = false;
            }
            cur = r;
#pragma unroll
            for (int k = 0; k < KV; ++k) {
              VecT x;
              if (ok[k]) x = *reinterpret_cast<const VecT *>(xr_base + r * W + lc[k]);
#pragma unroll
              for (int i = 0; i < VECW; ++i) {
                xr[k][i] = ok[k] ? to_acc<T>(x.v[i]) : A(0);
                acc[k][i] = A(0);
              }
            }
          }
#pragma unroll
          for (int k = 0; k < KV; ++k) {
            if (!ok[k]) continue;
#pragma unroll
            for (int i = 0; i < VECW; ++i) {
              const A uu = xr[k][i] + to_acc<T>(v[u][k].v[i]);
              const A gg = gv[u][k];
              acc[k][i] += uu > A(0) ? gg : gg * slope;
              aacc[k][i] += gg * leaky(uu, slope);
            }
          }
        }
      }
    }
    // the chunk's last run
    if (flags & FLAG_THROUGH) to_smem(s_head + warp * wc);
    else if (flags & FLAG_TAIL) to_smem(s_tail + warp * wc);
    else if (first && (flags & FLAG_HEAD)) to_smem(s_head + warp * wc);
    else store_row(cur, acc);
  }
  if (p.att_part) {
#pragma unroll
    for (int k = 0; k < KV; ++k)
      if (ok[k])
#pragma unroll
        for (int i = 0; i < VECW; ++i) s_att[warp * wc + lc[k] + i] = aacc[k][i];
  }
  __syncthreads();

  // ---- chains of pieces inside the tile, left to right ----
  if (cb < ce) {
    A a[KV][VECW];
    auto load_piece = [&](const A *src) {
#pragma unroll
      for (int k = 0; k < KV; ++k)
#pragma unroll
        for (int i = 0; i < VECW; ++i) a[k][i] = ok[k] ? src[lc[k] + i] : A(0);
    };
    auto add_piece = [&](const A *src) {
#pragma unroll
      for (int k = 0; k < KV; ++k)
#pragma unroll
        for (int i = 0; i < VECW; ++i)
          if (ok[k]) a[k][i] += src[lc[k] + i];
    };
    auto to_carry = [&](void *carry) {
      A *dst = static_cast<A *>(carry) + tile * wc;
#pragma unroll
      for (int k = 0; k < KV; ++k)
        if (ok[k])
#pragma unroll
          for (int i = 0; i < VECW; ++i) dst[lc[k] + i] = a[k][i];
    };
    if (warp == 0 && (flags & FLAG_HEAD)) {
      // the row that entered the tile from the left: its tile piece goes to the workspace
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
      if (inside) store_row(r1, a);
      else to_carry(p.carry_tail);      // the row goes on in the next tile
    }
  }
  if (p.att_part) {
    A *dst = static_cast<A *>(p.att_part) + tile * wc;
    for (int c = tid; c < wc; c += kThreads) {
      A s = s_att[c];
      for (int w = 1; w < kGvWarps; ++w) s += s_att[w * wc + c];
      dst[c] = s;
    }
  }
  if (tid == 0) {
    const bool through = t_head && t_cont && first_row == last_row;
    p.flags[tile] = (unsigned char)((t_head ? FLAG_HEAD : 0) | (through ? FLAG_THROUGH : 0) |
                                    ((t_cont && !through) ? FLAG_TAIL : 0));
  }
}

// A chain = tail[t] + head[t+1] + ... + head[last], last the first tile after t that is not THROUGH, added in that
// order; one warp per chain, lanes over the columns.  The sum times att is the row's gradient.
template <typename T>
__global__ void __launch_bounds__(kThreads) gatv2_fixup_kernel(const __grid_constant__ Gatv2GradParams p) {
  using A = typename AccOf<T>::type;
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
  const int wc = p.wc;
  const int64_t te = kGvWarps * (int64_t)p.chunk;
  const int64_t r = p.row_index[min((t + 1) * te, p.E) - 1];
  const A *head = static_cast<const A *>(p.carry_head);
  const A *tail = static_cast<const A *>(p.carry_tail);
  const T *att = static_cast<const T *>(p.att) + p.c0;
  T *out = static_cast<T *>(p.grad_row) + r * p.W + p.c0;
  for (int c = lane; c < wc; c += 32) {
    A a = tail[t * wc + c];
    for (int64_t j = t + 1; j <= last; ++j) a += head[j * wc + c];
    out[c] = from_acc<T>(to_acc<T>(att[c]) * a);
  }
}

// Rows of grad_row [S_out, W] that no edge reaches -- beyond the plan's rows, or with rowptr[r] == rowptr[r + 1] -- are
// zero.  One warp per row.
template <typename T>
__global__ void __launch_bounds__(kThreads) gatv2_zero_kernel(T *grad_row, const int64_t *rowptr, int64_t S_plan,
                                                              int64_t S_out, int64_t W) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t)gridDim.x * kThreads) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5; r < S_out; r += n_warps) {
    if (r < S_plan && rowptr[r] != rowptr[r + 1]) continue;
    for (int64_t c = lane; c < W; c += 32) grad_row[r * W + c] = from_acc<T>(0);
  }
}

// Column sums of in [n][wc] (accumulator type), rows in slices: block (x, y) adds rows [y n / gridDim.y, (y+1) n /
// gridDim.y) of columns [32 x, 32 x + 32) -- 8 row strides in sequence, then the strides in order.  The result goes to
// part [gridDim.y][wc], or rounded to out [wc] (one slice).
template <typename T>
__global__ void __launch_bounds__(kThreads) gatv2_att_kernel(const typename AccOf<T>::type *in, int64_t n, int wc,
                                                             typename AccOf<T>::type *part, T *out) {
  using A = typename AccOf<T>::type;
  __shared__ A s[kThreads / 32][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int64_t lo = n * blockIdx.y / gridDim.y, hi = n * (blockIdx.y + 1) / gridDim.y;
  A a = A(0);
  if (c < wc)
    for (int64_t i = lo + ty; i < hi; i += kThreads / 32) a += in[i * wc + c];
  s[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && c < wc) {
    for (int j = 1; j < kThreads / 32; ++j) a += s[j][tx];
    if (out) out[c] = from_acc<T>(a);
    else part[(int64_t)blockIdx.y * wc + c] = a;
  }
}

}  // namespace geot
