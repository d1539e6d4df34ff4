// sddmm.cuh -- sampled dense-dense product on a COO edge list, sm_100a, one dot product per edge and head:
//
//     out[e, h] = < mat1[row_index[e], h, :] , mat2[col_index[e], h, :] >   e = 0 .. E-1,  h = 0 .. H-1
//
// H = 1 is the weight gradient of gather_weight_scatter; H > 1 (rows of W = H*F elements) that of mh_spmm.
// Replaces the reference's sddmm_coo_ebalance_{vec4,vec2,scalar} (csrc/cuda/sddmm_coo_kernel.cuh:3-215,
// launcher csrc/cuda/gather_weight_scatter_cuda.cu:41-62), which serve the weight gradient of
// gather_weight_scatter (geot/gather_weight_scatter.py:47).  The reference is fp32 + int32 only and
// launches nnz/16 blocks of 32 threads; this one is built like segment_reduce_kernel:
//
//   * edge-count partition: a GROUP of LPR lanes owns `chunk_edges` consecutive edges and keeps whole
//     rows in registers (128-bit loads); a 256-thread CTA owns 256/LPR chunks;
//   * index streams are read once per edge, coalesced (lane l loads edge l of the batch), with an L2
//     evict-first policy; row offsets reach the other lanes by shuffle;
//   * row_index is the sorted one in the backward pass (dst-sorted edge list): the mat1 row stays in
//     registers while consecutive edges share it and is re-loaded only at a segment head -- half the
//     row traffic of the reference.  Sortedness is not required for correctness;
//   * indices are loaded two batches ahead; the gathered mat2 rows are staged through a per-group shared-memory
//     ring by cp.async (PF sub-batches of U rows in flight, as in segment_reduce_kernel), or -- narrow rows and
//     unaligned data -- double-buffered in registers;
//   * the U per-lane partial dot products are reduced across the group with a transposing butterfly
//     (U - 1 + log2(LPR/U) shuffles per U edges instead of U * log2(LPR)), after which lane k*(LPR/U)
//     holds edge k's result: U consecutive outputs = one 32-byte sector;
//   * H > 1: a head is HV whole vectors (HV a power of two).  With HV <= LPR the butterfly runs over the low log2(HV)
//     lane bits only and a lane keeps one partial per vector it holds (each of its VPL vectors is in another head);
//     the results are then gathered so that the LPR * H outputs of a batch leave in coalesced stores, as [E,H] (the
//     H results of an edge contiguous) or [H,E] (the edges of a head contiguous).
//   * OP: the elementwise step before the reduction over a head's columns.  SDDMM_DOT (the default) is a * b;
//     SDDMM_GATV2 is att[c] * leaky_relu(a + b) -- the GATv2 attention score with mat1 = x_r by dst, mat2 = x_l by src
//     (gatv2.cu).  a + b is formed in the accumulator, then the slope, then the product with att; one rounding on the
//     store.  A lane holds the same columns for every edge, so its att values are loaded once.
#pragma once
#include "segment_reduce.cuh"

namespace geot {

struct SddmmParams {
  const void *mat1;             // [N1, W], indexed by row_index
  const void *mat2;             // [N2, W], indexed by col_index
  const int64_t *row_index;     // [E]
  const int64_t *col_index;     // [E]
  void *out;                    // [E, H], or [H, E] with head_major
  int64_t E;
  int64_t W;                    // H * F
  int64_t H;
  int head_major;
  int chunk_edges;
};

// gatv2_score_kernel: the same operands, plus
struct Gatv2ScoreParams : SddmmParams {
  const void *att;              // [H, F] = [W], of the operands' type
  double slope;                 // leaky_relu negative slope
};

enum : int { SDDMM_DOT = 0, SDDMM_GATV2 = 1 };

// leaky_relu as torch computes it: u > 0 ? u : u * slope (NaN goes through the product)
template <typename A> __device__ __forceinline__ A leaky(A u, A slope) { return u > A(0) ? u : u * slope; }

// Transposing butterfly over the low log2(LPR) lane bits: p[0..U) per lane in.  On return, with U <= LPR, p[0] of lane
// gl holds the sum over its LPR lanes of value ((gl % LPR) / (LPR / U)); with U > LPR, p[0 .. U/LPR) hold values
// (gl % LPR) * (U / LPR) + 0 .. U/LPR-1.
template <int U, int LPR, typename A>
__device__ __forceinline__ void group_transpose_reduce(A (&p)[U], unsigned gmask, int gl) {
  int n = U;
#pragma unroll
  for (int s = LPR / 2; s >= 1; s >>= 1) {
    if (n > 1) {
      const bool up = (gl & s) != 0;
      const int h = n / 2;
#pragma unroll
      for (int i = 0; i < U / 2; ++i) {
        if (i < h) {
          const A send = up ? p[i] : p[i + h];
          const A keep = up ? p[i + h] : p[i];
          p[i] = keep + __shfl_xor_sync(gmask, send, s, 32);
        }
      }
      n = h;
    } else {
      p[0] += __shfl_xor_sync(gmask, p[0], s, 32);
    }
  }
}

// PF == 0: gathered mat2 rows go global -> registers, double buffered.  PF > 0: they are staged through a per-group
// shared-memory ring by cp.async exactly as in segment_reduce_kernel (PF sub-batches of U rows in flight).
// HV: vectors per head, a power of two; LPR * VPL is one head over the whole row (H = 1).
template <typename T, int VECW, int LPR, int VPL, int PF, int HV = LPR * VPL>
struct SddmmShape {
  static constexpr int NG = kThreads / LPR;
  static constexpr int R = HV < LPR ? HV : LPR;                 // lanes that share a head's partial sums
  static constexpr int HPJ = LPR / R;                           // heads in one vector layer j of the group
  static constexpr int NP = HV < LPR ? VPL : VPL * LPR / HV;    // partials per lane and edge: heads it touches
  static constexpr int NH = HPJ * NP;                           // heads the group holds
  static_assert(HV <= LPR || HV % LPR == 0, "a head is whole vector layers or a power-of-two lane group");
  static constexpr int CW = LPR * VPL * VECW;
  // (several heads over several vector layers: half the sub-batch, for registers)
  static constexpr int U0 = PF > 0 ? ((VPL >= 4 || (NH > 1 && VPL >= 2)) ? 2 : 4) : ((VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8));
  static constexpr int U = (LPR < U0) ? LPR : U0;
  static constexpr int NS = PF + 1;
  static constexpr size_t smem_bytes = PF > 0 ? (size_t)NG * NS * U * CW * sizeof(T) : 0;
  static constexpr int max_blocks = (int)((227 * 1024) / (smem_bytes + 1024));
  // (several heads: room for one result per head and the slot map of the collection below)
  static constexpr int min_blocks = (PF == 0 || NH > 1) ? 2 : (max_blocks >= 3 ? 3 : (max_blocks >= 2 ? 2 : 1));
  // SDDMM_GATV2 holds the lane's att columns too: one CTA fewer per SM, so that no shape spills
  static constexpr int min_blocks_of(int op) { return op == 0 ? min_blocks : min_blocks - 1; }
  static_assert(PF == 0 || PF * U <= LPR, "the prefetch distance must stay within one batch ahead");
};

// P: SddmmParams, or Gatv2ScoreParams for OP = SDDMM_GATV2.
template <typename T, int VECW, int LPR, int VPL, int PF, int HV = LPR * VPL, int OP = SDDMM_DOT, typename P = SddmmParams>
__global__ void __launch_bounds__(kThreads, (SddmmShape<T, VECW, LPR, VPL, PF, HV>::min_blocks_of(OP))) sddmm_coo_kernel(const P p) {
  using A = typename AccOf<T>::type;
  using VecT = Vec<T, VECW>;
  using SH = SddmmShape<T, VECW, LPR, VPL, PF, HV>;
  constexpr int NG = SH::NG, CW = SH::CW, U = SH::U, NS = SH::NS;
  constexpr int R = SH::R, HPJ = SH::HPJ, NP = SH::NP, NH = SH::NH;
  // after the butterfly over R lanes, value v = u * NP + q of the head group sits at lane (v / QV) * DV, slot v % QV
  constexpr int NV = U * NP, QV = NV > R ? NV / R : 1, DV = NV < R ? R / NV : 1;
  extern __shared__ __align__(16) unsigned char sddmm_smem[];

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int g = tid / LPR;
  const int gl = tid % LPR;
  const unsigned gmask = group_mask<LPR>(lane);
  const int gshift = lane & ~(LPR - 1);
  const int64_t E = p.E, W = p.W;
  const int C = p.chunk_edges;
  const int64_t e_begin = ((int64_t)blockIdx.x * NG + g) * (int64_t)C;
  const int64_t e_end = min(e_begin + (int64_t)C, E);
  if (e_begin >= e_end) return;     // whole groups leave together: no block-level barrier below
  const int64_t H = p.H;

  const T *__restrict__ mat1 = static_cast<const T *>(p.mat1);
  const T *__restrict__ mat2 = static_cast<const T *>(p.mat2);
  T *__restrict__ out = static_cast<T *>(p.out);
  const uint64_t pol = policy_evict_first();
  const int64_t row_bytes = W * (int64_t)sizeof(T);

  // This lane's columns; lanes past the row end read column 0 and contribute nothing.
  bool col_ok[VPL];
  int64_t col_b[VPL];   // byte offset of this lane's vector j inside a row
#pragma unroll
  for (int j = 0; j < VPL; ++j) {
    const int64_t c = (int64_t)(j * LPR + gl) * VECW;
    col_ok[j] = c < W;
    col_b[j] = (col_ok[j] ? c : 0) * (int64_t)sizeof(T);
  }
  const char *m1 = reinterpret_cast<const char *>(mat1);
  const char *m2 = reinterpret_cast<const char *>(mat2);
  [[maybe_unused]] A att[OP == SDDMM_GATV2 ? VPL : 1][OP == SDDMM_GATV2 ? VECW : 1];
  [[maybe_unused]] A slope = A(0);
  if constexpr (OP == SDDMM_GATV2) {
    slope = A(p.slope);
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const VecT v = *reinterpret_cast<const VecT *>(static_cast<const char *>(p.att) + col_b[j]);
#pragma unroll
      for (int i = 0; i < VECW; ++i) att[j][i] = to_acc<T>(v.v[i]);
    }
  }

  T *ring = nullptr;      // this group's ring; lane piece j of row r at r*CW + (j*LPR + gl)*VECW
  uint32_t ring_s = 0;
  if constexpr (PF > 0) {
    ring = reinterpret_cast<T *>(sddmm_smem) + (size_t)g * (NS * U * CW) + gl * VECW;
    ring_s = (uint32_t)__cvta_generic_to_shared(ring);
  }

  A a[VPL][VECW];   // the current mat1 row, as accumulator type, zero outside the row
#pragma unroll
  for (int j = 0; j < VPL; ++j)
#pragma unroll
    for (int i = 0; i < VECW; ++i) a[j][i] = A(0);

  auto load_a = [&](int64_t off1) {
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const VecT v = *reinterpret_cast<const VecT *>(m1 + off1 + col_b[j]);
#pragma unroll
      for (int i = 0; i < VECW; ++i) a[j][i] = col_ok[j] ? to_acc<T>(v.v[i]) : A(0);
    }
  };

  // batch operands of this lane: edge b + gl.  Edges past the chunk end alias edge e_end-1: valid
  // addresses, no extra segment heads, results never stored.
  auto load_idx = [&](int64_t b, int64_t &row, int64_t &off1, int64_t &off2) {
    const int64_t le = min(b + gl, e_end - 1);
    row = ld_stream(p.row_index + le, pol);
    off1 = row * row_bytes;
    off2 = ld_stream(p.col_index + le, pol) * row_bytes;
  };
  // U gathered mat2 rows of sub-batch [k0, k0+U) of a batch whose offsets are in `offs`: to registers ...
  auto load_v = [&](VecT(&v)[U][VPL], int64_t offs, int k0) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t off2 = __shfl_sync(gmask, offs, k0 + u, LPR);
#pragma unroll
      for (int j = 0; j < VPL; ++j) v[u][j] = *reinterpret_cast<const VecT *>(m2 + off2 + col_b[j]);
    }
  };
  // ... or into ring stage `stage`
  auto ring_issue = [&](int64_t offs, int k0, int stage) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t off2 = __shfl_sync(gmask, offs, k0 + u, LPR);
#pragma unroll
      for (int j = 0; j < VPL; ++j)
        cp_async_16(ring_s + (uint32_t)(((stage * U + u) * CW + j * LPR * VECW) * sizeof(T)), m2 + off2 + col_b[j]);
    }
  };

  // operands of the current batch (my_*) and the next (n_*); the one after is loaded at the top of each iteration
  int64_t my_row, my_off1, my_off2, n_row = 0, n_off1 = 0, n_off2 = 0;
  load_idx(e_begin, my_row, my_off1, my_off2);
  if (e_begin + LPR < e_end) load_idx(e_begin + LPR, n_row, n_off1, n_off2);
  VecT vc[U][VPL];                 // the sub-batch being consumed
  int stage = 0;
  if constexpr (PF > 0) {
#pragma unroll
    for (int q = 0; q < PF; ++q) {
      ring_issue(my_off2, q * U, q);
      cp_async_commit();
    }
  } else {
    load_v(vc, my_off2, 0);
  }
  int64_t last_row = -1;           // row_index of the edge left of the current batch (none yet: forces a load)

  // The outputs this lane stores per batch: slot i is (edge k of the batch, head h); [H,E]: edge gl, head i; [E,H]:
  // element gl + i * LPR of the batch's contiguous LPR * H outputs.  Per slot, 16 bits, two to a register: k (8 bits),
  // and where the butterfly leaves (k, h): position v % QV (3 bits) of lane src (5 bits).
  static_assert(NH <= 16 && QV <= 8, "slot fields");
  unsigned slot2[(NH + 1) / 2];
  if constexpr (NH > 1) {
#pragma unroll
    for (int i = 0; i < NH; ++i) {
      const int k = p.head_major ? gl : (gl + i * LPR) / (int)H;
      const int h = p.head_major ? i : gl + i * LPR - k * (int)H;
      const int v = (k % U) * NP + h / HPJ;
      const unsigned sl = (unsigned)((k << 8) | ((v % QV) << 5) | ((h % HPJ) * R + (v / QV) * DV));
      slot2[i / 2] = (i % 2) ? (slot2[i / 2] | (sl << 16)) : sl;
    }
  }
  auto slot = [&](int i) { return (int)((slot2[i / 2] >> ((i % 2) * 16)) & 0xffffu); };

  for (int64_t b = e_begin; b < e_end; b += LPR) {
    const bool has_next = b + LPR < e_end;
    int64_t nn_row = 0, nn_off1 = 0, nn_off2 = 0;
    if (b + 2 * LPR < e_end) load_idx(b + 2 * LPR, nn_row, nn_off1, nn_off2);

    int64_t left = __shfl_up_sync(gmask, my_row, 1, LPR);
    if (gl == 0) left = last_row;
    const unsigned bmask = (__ballot_sync(gmask, my_row != left) >> gshift) & low_bits<LPR>();
    last_row = __shfl_sync(gmask, my_row, LPR - 1, LPR);

    A mine[NH];      // results of this lane's output slots, collected from the sub-batches below
#pragma unroll
    for (int i = 0; i < NH; ++i) mine[i] = A(0);
#pragma unroll
    for (int k0 = 0; k0 < LPR; k0 += U) {
      VecT vn[U][VPL];
      if constexpr (PF > 0) {
        // keep PF sub-batches in flight, then wait for the oldest and read this lane's own pieces back
        const int kk = k0 + PF * U;
        int st = stage + PF;
        if (st >= NS) st -= NS;
        if (kk < LPR) ring_issue(my_off2, kk, st);
        else if (has_next) ring_issue(n_off2, kk - LPR, st);
        cp_async_commit();
        cp_async_wait<PF>();
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < VPL; ++j)
            vc[u][j] = *reinterpret_cast<const VecT *>(ring + ((stage * U + u) * CW + j * LPR * VECW));
        stage = (stage + 1 == NS) ? 0 : stage + 1;
      } else {
        // next sub-batch's rows leave before this one is reduced (this batch, else the next batch's first)
        if (k0 + U < LPR) load_v(vn, my_off2, k0 + U);
        else if (has_next) load_v(vn, n_off2, 0);
      }

      A part[NV];      // partial q of edge k0 + u at u * NP + q
      const unsigned sub = (bmask >> k0) & low_bits<U>();
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (sub != 0 && ((sub >> u) & 1u)) load_a(__shfl_sync(gmask, my_off1, k0 + u, LPR));
        A s[NP];
#pragma unroll
        for (int q = 0; q < NP; ++q) s[q] = A(0);
#pragma unroll
        for (int j = 0; j < VPL; ++j)
#pragma unroll
          for (int i = 0; i < VECW; ++i) {
            if constexpr (OP == SDDMM_GATV2) {
              // lanes past the row end hold no columns: nothing, not att * leaky of column 0
              if (col_ok[j]) s[HV < LPR ? j : j / (HV / LPR)] += att[j][i] * leaky(a[j][i] + to_acc<T>(vc[u][j].v[i]), slope);
            } else {
              s[HV < LPR ? j : j / (HV / LPR)] += a[j][i] * to_acc<T>(vc[u][j].v[i]);
            }
          }
#pragma unroll
        for (int q = 0; q < NP; ++q) part[u * NP + q] = s[q];
      }
      if constexpr (NH > 1) {
        // head h is partial h / HPJ of the lanes [(h % HPJ) * R, +R); lane gl collects its slots of this sub-batch
        group_transpose_reduce<NV, R, A>(part, gmask, gl);
#pragma unroll
        for (int i = 0; i < NH; ++i) {
          const int src = slot(i) & 31;
          A r = __shfl_sync(gmask, part[0], src, LPR);
#pragma unroll
          for (int q = 1; q < QV; ++q) {
            const A t = __shfl_sync(gmask, part[q], src, LPR);
            if (((slot(i) >> 5) & 7) == q) r = t;
          }
          if ((slot(i) >> 8) / U == k0 / U) mine[i] = r;
        }
      } else if constexpr (LPR > 1) {
        group_transpose_reduce<U, LPR, A>(part, gmask, gl);
        // value k sits in lanes [k*(LPR/U), (k+1)*(LPR/U)); lane gl wants edge gl = sub-batch gl/U, value gl%U
        const A r = __shfl_sync(gmask, part[0], (gl % U) * (LPR / U), LPR);
        if (gl / U == k0 / U) mine[0] = r;
      } else {
        mine[0] = part[0];
      }
      if constexpr (PF == 0) {
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < VPL; ++j) vc[u][j] = vn[u][j];
      }
    }
    if constexpr (NH == 1) {
      if (b + gl < e_end) out[b + gl] = from_acc<T>(mine[0]);
    } else {
#pragma unroll
      for (int i = 0; i < NH; ++i) {
        if (p.head_major) {
          if (i < H && b + gl < e_end) out[i * E + b + gl] = from_acc<T>(mine[i]);
        } else if (gl + i * LPR < LPR * H && b + (slot(i) >> 8) < e_end) {
          out[b * H + gl + i * LPR] = from_acc<T>(mine[i]);
        }
      }
    }
    my_row = n_row; my_off1 = n_off1; my_off2 = n_off2;
    n_row = nn_row; n_off1 = nn_off1; n_off2 = nn_off2;
  }
}

// Rows wider than a group can hold in registers (W > 32 lanes * 4 vectors), and heads without a lane mapping (not a
// power-of-two number of whole vectors, or more than the group holds): one warp per edge, heads and columns in loops.
// MH = false is the single-head (H = 1) instantiation.
template <typename T, bool MH, int OP = SDDMM_DOT, typename P = SddmmParams>
__global__ void __launch_bounds__(kThreads) sddmm_coo_wide_kernel(const P p) {
  using A = typename AccOf<T>::type;
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * kThreads) >> 5;
  const T *__restrict__ mat1 = static_cast<const T *>(p.mat1);
  const T *__restrict__ mat2 = static_cast<const T *>(p.mat2);
  T *__restrict__ out = static_cast<T *>(p.out);
  const int64_t H = MH ? p.H : 1, F = MH ? p.W / p.H : p.W;
  for (int64_t e = warp; e < p.E; e += n_warps) {
    const T *x = mat1 + p.row_index[e] * p.W;
    const T *y = mat2 + p.col_index[e] * p.W;
    for (int64_t h = 0; h < H; ++h) {
      A s = A(0);
      if constexpr (OP == SDDMM_GATV2) {
        const T *att = static_cast<const T *>(p.att);
        const A slope = A(p.slope);
        for (int64_t c = h * F + lane; c < (h + 1) * F; c += 32)
          s += to_acc<T>(att[c]) * leaky(to_acc<T>(x[c]) + to_acc<T>(y[c]), slope);
      } else {
        for (int64_t c = h * F + lane; c < (h + 1) * F; c += 32) s += to_acc<T>(x[c]) * to_acc<T>(y[c]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) out[!MH ? e : p.head_major ? h * p.E + e : e * H + h] = from_acc<T>(s);
    }
  }
}

}  // namespace geot
