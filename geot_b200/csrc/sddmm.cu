// sddmm.cu -- C-ABI entry geot_b200_sddmm_coo (include/geot_b200.h) and its kernel shape selection.
// Replaces sddmm_coo_cuda (csrc/cuda/header_cuda.h:19-21, csrc/cuda/gather_weight_scatter_cuda.cu:41-62).
#include <cuda_runtime.h>
#include <stdio.h>

#include "internal.h"
#include "kernels/sddmm.cuh"

namespace geot {
namespace {

template <typename T, int VECW, int LPR, int VPL>
cudaError_t launch_sddmm(SddmmParams p, cudaStream_t stream) {
  constexpr int NG = kThreads / LPR;
  // cp.async ring for 16-byte vectors and rows of >= 8 vectors: depth 3 for 256-byte rows, 2 otherwise
  constexpr int PF = (VECW * sizeof(T) == 16 && LPR >= 8) ? (LPR == 16 ? 3 : 2) : 0;
  using SH = SddmmShape<T, VECW, LPR, VPL, PF>;
  // edge-count partition: as segment_reduce (abi.cu choose_config) -- long chunks for large inputs,
  // shorter ones until the grid covers the 148 SMs a few times over
  int chunk = 256;
  while (chunk > LPR && chunk > 8 && (p.E + (int64_t)NG * chunk - 1) / ((int64_t)NG * chunk) < 8 * 148) chunk >>= 1;
  if (chunk < LPR) chunk = LPR;
  p.chunk_edges = chunk;
  const int64_t blocks = (p.E + (int64_t)NG * chunk - 1) / ((int64_t)NG * chunk);
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
  auto kern = sddmm_coo_kernel<T, VECW, LPR, VPL, PF>;
  if (SH::smem_bytes > 48 * 1024) {
    static bool configured[64] = {};   // per instantiation and device ordinal (the attribute is per device)
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SH::smem_bytes);
      if (e != cudaSuccess) return e;
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  kern<<<(unsigned)blocks, kThreads, SH::smem_bytes, stream>>>(p);
  return cudaGetLastError();
}

template <typename T, int VECW>
cudaError_t launch_sddmm_shape(const SddmmParams &p, cudaStream_t stream) {
  const int64_t nvec = (p.W + VECW - 1) / VECW;
  if (nvec <= 1) return launch_sddmm<T, VECW, 1, 1>(p, stream);
  if (nvec <= 2) return launch_sddmm<T, VECW, 2, 1>(p, stream);
  if (nvec <= 4) return launch_sddmm<T, VECW, 4, 1>(p, stream);
  if (nvec <= 8) return launch_sddmm<T, VECW, 8, 1>(p, stream);
  if (nvec <= 16) return launch_sddmm<T, VECW, 16, 1>(p, stream);
  if (nvec <= 32) return launch_sddmm<T, VECW, 32, 1>(p, stream);
  if (nvec <= 64) return launch_sddmm<T, VECW, 32, 2>(p, stream);
  if constexpr (VECW <= 4) {
    if (nvec <= 128) return launch_sddmm<T, VECW, 32, 4>(p, stream);
  }
  const int64_t warps_per_block = kThreads / 32;
  const int64_t blocks = (p.E + warps_per_block - 1) / warps_per_block;
  const unsigned grid = (unsigned)(blocks < 148 * 32 ? blocks : 148 * 32);
  sddmm_coo_wide_kernel<T><<<grid, kThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_sddmm_type(const SddmmParams &p, bool vector_ok, cudaStream_t stream) {
  constexpr int FULL = 16 / (int)sizeof(T);
  if (vector_ok && p.W % FULL == 0) return launch_sddmm_shape<T, FULL>(p, stream);
  return launch_sddmm_shape<T, 1>(p, stream);
}

}  // namespace
}  // namespace geot

extern "C" int geot_b200_sddmm_coo(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index,
                                   void *out, int64_t E, int64_t F, int dtype, cudaStream_t stream) {
  if (E < 0 || F <= 0 || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_OK;      // nothing to do (pointers of empty buffers may be null)
  if (!mat1 || !mat2 || !row_index || !col_index || !out) return GEOT_ERR_INVALID_ARG;
  geot::SddmmParams p;
  p.mat1 = mat1; p.mat2 = mat2; p.row_index = row_index; p.col_index = col_index; p.out = out;
  p.E = E; p.W = F; p.chunk_edges = 0;
  const bool aligned = ((reinterpret_cast<uintptr_t>(mat1) | reinterpret_cast<uintptr_t>(mat2)) & 15) == 0;
  cudaError_t e;
  switch (dtype) {
    case GEOT_F32: e = geot::launch_sddmm_type<float>(p, aligned, stream); break;
    case GEOT_F64: e = geot::launch_sddmm_type<double>(p, aligned, stream); break;
    case GEOT_BF16: e = geot::launch_sddmm_type<__nv_bfloat16>(p, aligned, stream); break;
    default: e = geot::launch_sddmm_type<__half>(p, aligned, stream); break;
  }
  if (e != cudaSuccess) return cuda_fail(e, "sddmm_coo launch");
  return GEOT_OK;
}
