// gatv2.cu -- C-ABI entries geot_b200_gatv2_score, geot_b200_gatv2_grad_workspace_bytes and geot_b200_gatv2_grad
// (include/geot_b200.h): the GATv2 attention score of every edge and its deterministic backward.  The score runs on the
// SDDMM launcher (sddmm.cu) with the GATv2 elementwise step; the backward's kernels and partition: kernels/gatv2.cuh.
#include <cuda_runtime.h>

#include "internal.h"
#include "kernels/gatv2.cuh"

namespace geot {
namespace {

struct GvLayout {
  int chunk;
  int64_t n_tiles;
  int slab;             // most columns of one launch
  size_t carry_bytes;   // one [n_tiles][min(W, slab)] accumulator array
  size_t part_bytes;    // [kGvAttSlices][min(W, slab)]
  size_t bytes;         // carry_head, carry_tail, att_part, the second-level att partials, flags
};

// The partition depends on E alone (the summation order, and so the bits of the result, too): long chunks for large
// inputs, shorter ones until the grid covers the 148 SMs a few times over.
GvLayout gv_layout(int64_t E, int64_t W, int dtype) {
  GvLayout l;
  int chunk = 256;
  while (chunk > 32 && (E + (int64_t)kGvWarps * chunk - 1) / ((int64_t)kGvWarps * chunk) < 8 * 148) chunk >>= 1;
  l.chunk = chunk;
  l.n_tiles = (E + (int64_t)kGvWarps * chunk - 1) / ((int64_t)kGvWarps * chunk);
  const size_t acc = dtype == GEOT_F64 ? 8 : 4;
  l.slab = dtype == GEOT_F64 ? gv_slab<double>() : gv_slab<float>();
  const size_t wc = (size_t)(W < l.slab ? W : l.slab);
  l.carry_bytes = align256((size_t)l.n_tiles * wc * acc);
  l.part_bytes = align256((size_t)kGvAttSlices * wc * acc);
  l.bytes = 3 * l.carry_bytes + l.part_bytes + align256((size_t)l.n_tiles);
  return l;
}

template <typename T, int VECW, int KV>
cudaError_t launch_grad_slab(const Gatv2GradParams &p, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  const size_t smem = 3 * (size_t)kGvWarps * p.wc * sizeof(A);
  gatv2_grad_kernel<T, VECW, KV><<<(unsigned)p.n_tiles, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_grad(Gatv2GradParams p, const GvLayout &l, bool vector_ok, T *grad_att, const geot_plan_t *plan,
                        int64_t S_out, char *ws, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  constexpr int FULL = 16 / (int)sizeof(T);
  cudaError_t e = cudaSuccess;
  // rows without edges first: the kernels below write every other row
  {
    const int64_t blocks = (S_out + kThreads / 32 - 1) / (kThreads / 32);
    gatv2_zero_kernel<T><<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), kThreads, 0, stream>>>(
        static_cast<T *>(p.grad_row), plan->rowptr, plan->S, S_out, p.W);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  A *part = reinterpret_cast<A *>(ws + 3 * l.carry_bytes);
  for (int64_t c0 = 0; c0 < p.W; c0 += l.slab) {
    p.c0 = c0;
    p.wc = (int)(p.W - c0 < l.slab ? p.W - c0 : l.slab);
    if (vector_ok) {
      const int nvec = (p.wc + FULL - 1) / FULL;
      if (nvec <= 32) e = launch_grad_slab<T, FULL, 1>(p, stream);
      else if constexpr (FULL <= 4) e = launch_grad_slab<T, FULL, 2>(p, stream);   // (16-bit types: 32 vectors a slab)
    } else {
      if (p.wc <= 32) e = launch_grad_slab<T, 1, 1>(p, stream);
      else if (p.wc <= 64) e = launch_grad_slab<T, 1, 2>(p, stream);
      else if (p.wc <= 128) e = launch_grad_slab<T, 1, 4>(p, stream);
      else if constexpr (sizeof(A) == 4) e = launch_grad_slab<T, 1, 8>(p, stream);
    }
    if (e != cudaSuccess) return e;
    const int64_t fix_blocks = (p.n_tiles + kThreads / 32 - 1) / (kThreads / 32);
    gatv2_fixup_kernel<T><<<(unsigned)fix_blocks, kThreads, 0, stream>>>(p);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (grad_att) {
      const unsigned gx = (unsigned)((p.wc + 31) / 32);
      const int64_t slices = p.n_tiles < kGvAttSlices ? p.n_tiles : kGvAttSlices;
      gatv2_att_kernel<T><<<dim3(gx, (unsigned)slices), kThreads, 0, stream>>>(
          static_cast<const A *>(p.att_part), p.n_tiles, p.wc, part, nullptr);
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
      gatv2_att_kernel<T><<<dim3(gx, 1), kThreads, 0, stream>>>(part, slices, p.wc, nullptr, grad_att + c0);
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
  }
  return cudaSuccess;
}

bool bad_shape(int64_t E, int64_t H, int64_t F, int dtype) {
  return E < 0 || H < 1 || F < 1 || F > INT64_MAX / H || dtype < GEOT_F32 || dtype > GEOT_F16 ||
         (E > 0 && H * F > INT64_MAX / E);
}

uintptr_t addr(const void *p) { return reinterpret_cast<uintptr_t>(p); }

}  // namespace
}  // namespace geot

extern "C" int geot_b200_gatv2_score(const void *x_l, const void *x_r, const void *att, const int64_t *src_index,
                                     const int64_t *dst_index, void *out, int64_t E, int64_t H, int64_t F, int dtype,
                                     const double *negative_slope, cudaStream_t stream) {
  if (!x_l || !x_r || !att || !src_index || !dst_index || !out || !negative_slope) return GEOT_ERR_INVALID_ARG;
  if (geot::bad_shape(E, H, F, dtype)) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_ERR_EMPTY;
  // mat1 = x_r by dst (held in registers while dst repeats), mat2 = x_l by src (through the ring)
  return geot::sddmm(x_r, dst_index, x_l, src_index, out, E, H, F, dtype, 0, stream, att, *negative_slope);
}

extern "C" size_t geot_b200_gatv2_grad_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype) {
  if (E <= 0 || geot::bad_shape(E, H, F, dtype)) return 256;
  return geot::gv_layout(E, H * F, dtype).bytes;
}

extern "C" int geot_b200_gatv2_grad(const void *x_row, const void *x_gat, const void *att, const void *grad_score,
                                    const int64_t *row_index, const int64_t *gat_index, const geot_plan_t *plan,
                                    int64_t S_out, void *grad_row, void *grad_att, int64_t E, int64_t H, int64_t F,
                                    int dtype, const double *negative_slope, void *workspace, size_t workspace_bytes,
                                    cudaStream_t stream) {
  // arguments, then E, then the plan, then the workspace; no CUDA call before all pass
  if (!x_row || !x_gat || !att || !grad_score || !row_index || !gat_index || !plan || !grad_row || !negative_slope ||
      !workspace)
    return GEOT_ERR_INVALID_ARG;
  if (geot::bad_shape(E, H, F, dtype) || S_out < 0) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_ERR_EMPTY;
  if (!plan->is_sorted || plan->E != E || !plan->rowptr || plan->max_row >= S_out)
    return GEOT_ERR_INVALID_ARG;
  const int64_t W = H * F;
  const geot::GvLayout l = geot::gv_layout(E, W, dtype);
  if ((geot::addr(workspace) & 255) || workspace_bytes < l.bytes) return GEOT_ERR_WORKSPACE;
  if (l.n_tiles > 0x7fffffffLL) return GEOT_ERR_UNSUPPORTED;

  char *ws = static_cast<char *>(workspace);
  geot::Gatv2GradParams p;
  p.x_row = x_row; p.x_gat = x_gat; p.att = att; p.grad = grad_score;
  p.row_index = row_index; p.gat_index = gat_index; p.grad_row = grad_row;
  p.E = E; p.W = W; p.H = H; p.F = F; p.c0 = 0; p.wc = 0; p.chunk = l.chunk; p.n_tiles = l.n_tiles;
  p.slope = *negative_slope;
  p.carry_head = ws;
  p.carry_tail = ws + l.carry_bytes;
  p.att_part = grad_att ? ws + 2 * l.carry_bytes : nullptr;
  p.flags = reinterpret_cast<unsigned char *>(ws + 3 * l.carry_bytes + l.part_bytes);
  const size_t es = dtype_size(dtype);
  // 16-byte vectors: whole vectors per head and aligned rows
  const bool vector_ok = (F * (int64_t)es) % 16 == 0 &&
                         ((geot::addr(x_row) | geot::addr(x_gat) | geot::addr(att) | geot::addr(grad_row)) & 15) == 0;
  cudaError_t e;
  switch (dtype) {
    case GEOT_F32:
      e = geot::launch_grad<float>(p, l, vector_ok, static_cast<float *>(grad_att), plan, S_out, ws, stream);
      break;
    case GEOT_F64:
      e = geot::launch_grad<double>(p, l, vector_ok, static_cast<double *>(grad_att), plan, S_out, ws, stream);
      break;
    case GEOT_BF16:
      e = geot::launch_grad<__nv_bfloat16>(p, l, vector_ok, static_cast<__nv_bfloat16 *>(grad_att), plan, S_out, ws,
                                           stream);
      break;
    default:
      e = geot::launch_grad<__half>(p, l, vector_ok, static_cast<__half *>(grad_att), plan, S_out, ws, stream);
      break;
  }
  if (e != cudaSuccess) return cuda_fail(e, "gatv2_grad launch");
  return GEOT_OK;
}
