// softmax.cu -- C-ABI entries geot_b200_segment_softmax{,_workspace_bytes,_backward} (include/geot_b200.h): the
// softmax of [E, H] edge logits over the edges of each dst row of a sorted edge list, and its backward.  Kernels and
// partition: kernels/softmax.cuh.
#include <cuda_runtime.h>

#include "internal.h"
#include "kernels/softmax.cuh"

namespace geot {
namespace {

struct SmLayout {
  int hp, nc;
  int64_t n_tiles;
  size_t carry_bytes;   // one [n_tiles][H] SmPair array
  size_t bytes;         // carry_head, carry_tail, stat_head, stat_tail, flags
};

// The partition depends on (E, H) alone: the combine order, and so the bits of the result, too.
SmLayout sm_layout(int64_t E, int64_t H, int dtype) {
  SmLayout l;
  l.hp = (int)(H < kThreads ? H : kThreads);
  l.nc = kThreads / l.hp;
  const int64_t te = (int64_t)l.nc * kSmChunk;
  l.n_tiles = (E + te - 1) / te;
  const size_t pair = 2 * (dtype == GEOT_F64 ? 8 : 4);
  l.carry_bytes = align256((size_t)l.n_tiles * (size_t)H * pair);
  l.bytes = 4 * l.carry_bytes + align256((size_t)l.n_tiles);
  return l;
}

template <typename T, bool BWD>
cudaError_t launch_softmax(SoftmaxParams p, cudaStream_t stream) {
  segment_softmax_kernel<T, BWD><<<(unsigned)p.n_tiles, kThreads, 0, stream>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int64_t fix_blocks = (p.n_tiles + kThreads / 32 - 1) / (kThreads / 32);
  segment_softmax_fixup_kernel<T, BWD><<<(unsigned)fix_blocks, kThreads, 0, stream>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  segment_softmax_finish_kernel<T, BWD><<<(unsigned)p.n_tiles, kThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

// Validation shared by both entries, in the order of the other device entries: arguments, then E, then the plan,
// then the workspace.  No CUDA call before it passes.
int check_args(bool pointers_ok, int64_t E, int64_t H, int dtype, const geot_plan_t *plan, const void *workspace,
               size_t workspace_bytes) {
  if (!pointers_ok || !plan || !workspace) return GEOT_ERR_INVALID_ARG;
  if (H < 1 || H > 0x7fffffff || E < 0 || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_ERR_EMPTY;
  if (H > INT64_MAX / E) return GEOT_ERR_INVALID_ARG;
  if (!plan->is_sorted || plan->E != E) return GEOT_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) || workspace_bytes < sm_layout(E, H, dtype).bytes)
    return GEOT_ERR_WORKSPACE;
  return GEOT_OK;
}

int softmax(const void *x, const void *g, const int64_t *dst_index, void *y, int64_t E, int64_t H, int dtype,
            void *workspace, cudaStream_t stream, bool bwd) {
  const SmLayout l = sm_layout(E, H, dtype);
  if (l.n_tiles > 0x7fffffffLL) return GEOT_ERR_UNSUPPORTED;
  char *ws = static_cast<char *>(workspace);
  SoftmaxParams p;
  p.x = x; p.g = g; p.dst_index = dst_index; p.y = y;
  p.E = E; p.H = (int)H; p.hp = l.hp; p.nc = l.nc; p.n_tiles = l.n_tiles;
  p.carry_head = ws;
  p.carry_tail = ws + l.carry_bytes;
  p.stat_head = ws + 2 * l.carry_bytes;
  p.stat_tail = ws + 3 * l.carry_bytes;
  p.flags = reinterpret_cast<unsigned char *>(ws + 4 * l.carry_bytes);
  cudaError_t e;
  switch (dtype) {
    case GEOT_F32: e = bwd ? launch_softmax<float, true>(p, stream) : launch_softmax<float, false>(p, stream); break;
    case GEOT_F64: e = bwd ? launch_softmax<double, true>(p, stream) : launch_softmax<double, false>(p, stream); break;
    case GEOT_BF16:
      e = bwd ? launch_softmax<__nv_bfloat16, true>(p, stream) : launch_softmax<__nv_bfloat16, false>(p, stream);
      break;
    default: e = bwd ? launch_softmax<__half, true>(p, stream) : launch_softmax<__half, false>(p, stream); break;
  }
  if (e != cudaSuccess) return cuda_fail(e, bwd ? "segment_softmax_backward launch" : "segment_softmax launch");
  return GEOT_OK;
}

}  // namespace
}  // namespace geot

extern "C" size_t geot_b200_segment_softmax_workspace_bytes(int64_t E, int64_t H, int dtype) {
  if (E <= 0 || H <= 0 || H > INT64_MAX / E || dtype < GEOT_F32 || dtype > GEOT_F16) return 256;
  return geot::sm_layout(E, H, dtype).bytes;
}

extern "C" int geot_b200_segment_softmax(const void *src, const int64_t *dst_index, void *out, int64_t E, int64_t H,
                                         int dtype, const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                                         cudaStream_t stream) {
  const int st = geot::check_args(src && dst_index && out, E, H, dtype, plan, workspace, workspace_bytes);
  if (st != GEOT_OK) return st;
  return geot::softmax(src, nullptr, dst_index, out, E, H, dtype, workspace, stream, false);
}

extern "C" int geot_b200_segment_softmax_backward(const void *out, const void *grad_out, const int64_t *dst_index,
                                                  void *grad_src, int64_t E, int64_t H, int dtype,
                                                  const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                                                  cudaStream_t stream) {
  const int st = geot::check_args(out && grad_out && dst_index && grad_src, E, H, dtype, plan, workspace, workspace_bytes);
  if (st != GEOT_OK) return st;
  return geot::softmax(out, grad_out, dst_index, grad_src, E, H, dtype, workspace, stream, true);
}
