// attention.cu -- C-ABI entries geot_b200_graph_attention{,_workspace_bytes} and geot_b200_graph_attention_grad{,
// _workspace_bytes} (include/geot_b200.h): fused dot-product graph attention and the dst pass of its backward.  Kernels
// and partition: kernels/attention.cuh.
#include <cuda_runtime.h>

#include "internal.h"
#include "kernels/attention.cuh"

namespace geot {
namespace {

struct AttLayout {
  int chunk;
  int64_t n_tiles;
  int slab;             // most columns of one launch
  size_t carry_bytes;   // one [n_tiles][piece] accumulator array
  size_t bytes;         // forward: carry_head, carry_tail, flags; backward: the same and the all-ones [W] factor
};

// The partition depends on E alone, as gv_layout (gatv2.cu).  A forward piece is [wc] acc, [hc] m and [hc] s; a
// launch holds hc whole heads of F columns, hc * F <= min(W, slab).  The backward piece is [wc].
AttLayout att_layout(int64_t E, int64_t H, int64_t F, int dtype, bool backward) {
  AttLayout l;
  int chunk = 256;
  while (chunk > 32 && (E + (int64_t)kGvWarps * chunk - 1) / ((int64_t)kGvWarps * chunk) < 8 * 148) chunk >>= 1;
  l.chunk = chunk;
  l.n_tiles = (E + (int64_t)kGvWarps * chunk - 1) / ((int64_t)kGvWarps * chunk);
  const size_t acc = dtype == GEOT_F64 ? 8 : 4;
  l.slab = dtype == GEOT_F64 ? gv_slab<double>() : gv_slab<float>();
  const int64_t W = H * F;
  const size_t wc = (size_t)(W < l.slab ? W : l.slab);
  const size_t piece = backward ? wc : wc + 2 * (wc / (size_t)F);
  l.carry_bytes = align256((size_t)l.n_tiles * piece * acc);
  l.bytes = 2 * l.carry_bytes + align256((size_t)l.n_tiles);
  if (backward) l.bytes += align256((size_t)W * dtype_size(dtype));
  return l;
}

// The lane mapping of a head of F columns: G lanes and VPH vectors of VECW columns per lane, both powers of two (the
// kernels are instantiated for those; slots past the head's last vector are masked off).  For F <= gv_slab(), VPH <=
// att_kv_max, itself a power of two.
struct AttMap {
  int G, vph;
};
AttMap att_map(int64_t F, int vecw) {
  const int64_t nv = (F + vecw - 1) / vecw;
  int G = 1;
  while (G < 32 && G < nv) G <<= 1;
  int vph = 1;
  while ((int64_t)vph * G < nv) vph <<= 1;
  return {G, vph};
}

template <typename T, int VECW, int NL, int VPH, bool BWD>
cudaError_t launch_slab(const AttentionParams &p, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  const int wc = p.hc * (int)p.F;
  const size_t smem = 2 * (size_t)kGvWarps * (BWD ? wc : wc + 2 * p.hc) * sizeof(A);
  auto kern = BWD ? attention_grad_kernel<T, VECW, NL, VPH> : attention_fwd_kernel<T, VECW, NL, VPH>;
  if (smem > 32 * 1024) {
    // past the default limit (48 KB less the kernel's static shared memory) the launch needs the opt-in
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e == cudaSuccess && smem > (size_t)fa.maxDynamicSharedSizeBytes)
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<(unsigned)p.n_tiles, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

// NL (layers) and VPH (vectors per head) as template arguments, both powers of two with NL * VPH <= att_kv_max
template <typename T, int VECW, int VPH, bool BWD, int NL = 1>
cudaError_t launch_nl(int nl, const AttentionParams &p, cudaStream_t stream) {
  if constexpr (NL * VPH <= att_kv_max<typename AccOf<T>::type, VECW>()) {
    if (nl == NL) return launch_slab<T, VECW, NL, VPH, BWD>(p, stream);
    return launch_nl<T, VECW, VPH, BWD, NL * 2>(nl, p, stream);
  } else {
    return cudaErrorInvalidValue;
  }
}
template <typename T, int VECW, bool BWD, int VPH = 1>
cudaError_t launch_vph(int vph, int nl, const AttentionParams &p, cudaStream_t stream) {
  if constexpr (VPH <= att_kv_max<typename AccOf<T>::type, VECW>()) {
    if (vph == VPH) return launch_nl<T, VECW, VPH, BWD>(nl, p, stream);
    return launch_vph<T, VECW, BWD, VPH * 2>(vph, nl, p, stream);
  } else {
    return cudaErrorInvalidValue;
  }
}

// Whole heads per launch: as many as the lanes hold (32 / G per layer, att_kv_max / VPH layers).
template <typename T>
cudaError_t launch(AttentionParams p, bool vector_ok, bool backward, const geot_plan_t *plan, int64_t N_dst,
                   cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  constexpr int FULL = 16 / (int)sizeof(T);
  const int vecw = vector_ok ? FULL : 1;
  const AttMap mp = att_map(p.F, vecw);
  const int kv_max = vector_ok ? att_kv_max<A, FULL>() : att_kv_max<A, 1>();
  const int hpl = 32 / mp.G;
  const int64_t per_launch = (int64_t)hpl * (kv_max / mp.vph);
  p.G = mp.G;
  cudaError_t e = cudaSuccess;
  for (int64_t h0 = 0; h0 < p.H; h0 += per_launch) {
    p.h0 = h0;
    p.hc = (int)(p.H - h0 < per_launch ? p.H - h0 : per_launch);
    int nl = 1;
    while (nl * hpl < p.hc) nl <<= 1;
    if (vector_ok) e = backward ? launch_vph<T, FULL, true>(mp.vph, nl, p, stream) : launch_vph<T, FULL, false>(mp.vph, nl, p, stream);
    else e = backward ? launch_vph<T, 1, true>(mp.vph, nl, p, stream) : launch_vph<T, 1, false>(mp.vph, nl, p, stream);
    if (e != cudaSuccess) return e;
    const unsigned fix_blocks = (unsigned)((p.n_tiles + kThreads / 32 - 1) / (kThreads / 32));
    if (backward) {
      // grad_q of the rows cut by tile boundaries: plain sums times the all-ones factor.  The fixup reads row_index,
      // grad_row, E, W, c0, wc, chunk, n_tiles, the carries, flags and att; x_row, x_gat, gat_index, grad, H, F,
      // slope and att_part are unused there.
      Gatv2GradParams g;
      g.x_row = g.x_gat = g.grad = nullptr;
      g.row_index = p.dst_index; g.gat_index = p.src_index; g.grad_row = p.out;
      g.E = p.E; g.W = p.W; g.H = p.H; g.F = p.F; g.c0 = h0 * p.F; g.wc = p.hc * (int)p.F; g.chunk = p.chunk;
      g.n_tiles = p.n_tiles; g.slope = 0.0; g.carry_head = p.carry_head; g.carry_tail = p.carry_tail;
      g.att_part = nullptr; g.flags = p.flags;
      g.att = reinterpret_cast<const char *>(p.flags) + align256((size_t)p.n_tiles);   // [W] ones (backward())
      gatv2_fixup_kernel<T><<<fix_blocks, kThreads, 0, stream>>>(g);
    } else {
      attention_fixup_kernel<T><<<fix_blocks, kThreads, 0, stream>>>(p);
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

bool bad_shape(int64_t E, int64_t H, int64_t F, int dtype) {
  return E < 0 || H < 1 || F < 1 || F > INT64_MAX / H || dtype < GEOT_F32 || dtype > GEOT_F16 ||
         (E > 0 && H * F > INT64_MAX / E);
}

uintptr_t addr(const void *p) { return reinterpret_cast<uintptr_t>(p); }

// the checks both entries share after their own null checks: E, the plan, the workspace, what the kernels support
int check_call(int64_t E, int64_t H, int64_t F, int dtype, const geot_plan_t *plan, int64_t N_dst, void *workspace,
               size_t workspace_bytes, bool backward, AttLayout *l) {
  if (bad_shape(E, H, F, dtype) || N_dst < 0) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_ERR_EMPTY;
  if (!plan->is_sorted || plan->E != E || !plan->rowptr || plan->max_row >= N_dst) return GEOT_ERR_INVALID_ARG;
  *l = att_layout(E, H, F, dtype, backward);
  if ((addr(workspace) & 255) || workspace_bytes < l->bytes) return GEOT_ERR_WORKSPACE;
  if (F > l->slab || l->n_tiles > 0x7fffffffLL) return GEOT_ERR_UNSUPPORTED;   // a head wider than one launch
  return GEOT_OK;
}

template <typename T>
cudaError_t forward(const AttentionParams &p, bool vector_ok, const geot_plan_t *plan, int64_t N_dst,
                    cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  // rows without edges first: the kernels below write every other row
  const int64_t blocks = (N_dst + kThreads / 32 - 1) / (kThreads / 32);
  if (N_dst > 0) {
    attention_empty_kernel<T><<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), kThreads, 0, stream>>>(
        static_cast<T *>(p.out), static_cast<A *>(p.lse), plan->rowptr, plan->S, N_dst, p.W, p.H);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return launch<T>(p, vector_ok, false, plan, N_dst, stream);
}

template <typename T>
cudaError_t backward(const AttentionParams &p, bool vector_ok, const geot_plan_t *plan, int64_t N_dst,
                     cudaStream_t stream) {
  const int64_t blocks = (N_dst + kThreads / 32 - 1) / (kThreads / 32);
  if (N_dst > 0) {
    gatv2_zero_kernel<T><<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), kThreads, 0, stream>>>(
        static_cast<T *>(p.out), plan->rowptr, plan->S, N_dst, p.W);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  T *ones = reinterpret_cast<T *>(reinterpret_cast<char *>(p.flags) + align256((size_t)p.n_tiles));
  const int64_t fb = (p.W + kThreads - 1) / kThreads;
  attention_fill_kernel<T><<<(unsigned)(fb < 148 ? fb : 148), kThreads, 0, stream>>>(ones, p.W, 1.0f);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return launch<T>(p, vector_ok, true, plan, N_dst, stream);
}

template <bool BWD>
cudaError_t dispatch(const AttentionParams &p, int dtype, bool vector_ok, const geot_plan_t *plan, int64_t N_dst,
                     cudaStream_t stream) {
  switch (dtype) {
    case GEOT_F32: return BWD ? backward<float>(p, vector_ok, plan, N_dst, stream) : forward<float>(p, vector_ok, plan, N_dst, stream);
    case GEOT_F64: return BWD ? backward<double>(p, vector_ok, plan, N_dst, stream) : forward<double>(p, vector_ok, plan, N_dst, stream);
    case GEOT_BF16:
      return BWD ? backward<__nv_bfloat16>(p, vector_ok, plan, N_dst, stream)
                 : forward<__nv_bfloat16>(p, vector_ok, plan, N_dst, stream);
    default: return BWD ? backward<__half>(p, vector_ok, plan, N_dst, stream) : forward<__half>(p, vector_ok, plan, N_dst, stream);
  }
}

}  // namespace
}  // namespace geot

extern "C" size_t geot_b200_graph_attention_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype) {
  if (E <= 0 || geot::bad_shape(E, H, F, dtype)) return 256;
  return geot::att_layout(E, H, F, dtype, false).bytes;
}

extern "C" int geot_b200_graph_attention(const void *q, const void *k, const void *v, const int64_t *src_index,
                                         const int64_t *dst_index, const geot_plan_t *plan, int64_t N_dst, void *out,
                                         void *lse, int64_t E, int64_t H, int64_t F, int dtype, const double *scale,
                                         void *workspace, size_t workspace_bytes, cudaStream_t stream) {
  // arguments, then E, then the plan, then the workspace; no CUDA call before all pass
  if (!q || !k || !v || !src_index || !dst_index || !plan || !out || !lse || !scale || !workspace)
    return GEOT_ERR_INVALID_ARG;
  geot::AttLayout l;
  const int st = geot::check_call(E, H, F, dtype, plan, N_dst, workspace, workspace_bytes, false, &l);
  if (st != GEOT_OK) return st;
  char *ws = static_cast<char *>(workspace);
  geot::AttentionParams p = {};
  p.q = q; p.k = k; p.v = v; p.src_index = src_index; p.dst_index = dst_index; p.out = out; p.lse = lse;
  p.E = E; p.W = H * F; p.H = H; p.F = F; p.chunk = l.chunk; p.n_tiles = l.n_tiles; p.scale = *scale;
  p.carry_head = ws;
  p.carry_tail = ws + l.carry_bytes;
  p.flags = reinterpret_cast<unsigned char *>(ws + 2 * l.carry_bytes);
  // 16-byte vectors: whole vectors per head and aligned rows
  const bool vector_ok = (F * (int64_t)dtype_size(dtype)) % 16 == 0 &&
                         ((geot::addr(q) | geot::addr(k) | geot::addr(v) | geot::addr(out)) & 15) == 0;
  const cudaError_t e = geot::dispatch<false>(p, dtype, vector_ok, plan, N_dst, stream);
  if (e != cudaSuccess) return cuda_fail(e, "graph_attention launch");
  return GEOT_OK;
}

extern "C" size_t geot_b200_graph_attention_grad_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype) {
  if (E <= 0 || geot::bad_shape(E, H, F, dtype)) return 256;
  return geot::att_layout(E, H, F, dtype, true).bytes;
}

extern "C" int geot_b200_graph_attention_grad(const void *q, const void *k, const void *v, const void *out,
                                              const void *lse, const void *grad_out, const int64_t *src_index,
                                              const int64_t *dst_index, const geot_plan_t *plan, int64_t N_dst,
                                              void *grad_q, void *p_out, void *ds_out, int64_t E, int64_t H, int64_t F,
                                              int dtype, const double *scale, void *workspace, size_t workspace_bytes,
                                              cudaStream_t stream) {
  if (!q || !k || !v || !out || !lse || !grad_out || !src_index || !dst_index || !plan || !grad_q || !p_out || !ds_out ||
      !scale || !workspace)
    return GEOT_ERR_INVALID_ARG;
  geot::AttLayout l;
  const int st = geot::check_call(E, H, F, dtype, plan, N_dst, workspace, workspace_bytes, true, &l);
  if (st != GEOT_OK) return st;
  char *ws = static_cast<char *>(workspace);
  geot::AttentionParams p = {};
  p.q = q; p.k = k; p.v = v; p.src_index = src_index; p.dst_index = dst_index; p.out = grad_q;
  p.lse = const_cast<void *>(lse); p.o = out; p.g = grad_out; p.p_out = p_out; p.ds_out = ds_out;
  p.E = E; p.W = H * F; p.H = H; p.F = F; p.chunk = l.chunk; p.n_tiles = l.n_tiles; p.scale = *scale;
  p.carry_head = ws;
  p.carry_tail = ws + l.carry_bytes;
  p.flags = reinterpret_cast<unsigned char *>(ws + 2 * l.carry_bytes);
  const bool vector_ok = (F * (int64_t)dtype_size(dtype)) % 16 == 0 &&
                         ((geot::addr(q) | geot::addr(k) | geot::addr(v) | geot::addr(out) | geot::addr(grad_out) |
                           geot::addr(grad_q)) & 15) == 0;
  const cudaError_t e = geot::dispatch<true>(p, dtype, vector_ok, plan, N_dst, stream);
  if (e != cudaSuccess) return cuda_fail(e, "graph_attention_grad launch");
  return GEOT_OK;
}
