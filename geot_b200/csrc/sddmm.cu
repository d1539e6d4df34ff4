// sddmm.cu -- C-ABI entries geot_b200_sddmm_coo and geot_b200_sddmm_mh (include/geot_b200.h) and their kernel shape
// selection; the same launcher runs the GATv2 attention score (att != null: geot_b200_gatv2_score, gatv2.cu).  geot_b200_sddmm_coo replaces sddmm_coo_cuda (csrc/cuda/header_cuda.h:19-21,
// csrc/cuda/gather_weight_scatter_cuda.cu:41-62); it is the H = 1 case of the multi-head launcher.
#include <cuda_runtime.h>
#include <stdio.h>

#include "internal.h"
#include "kernels/sddmm.cuh"

namespace geot {
namespace {

// Most heads a lane group keeps results for (one register per head and lane), and most bytes of per-lane results
// times vector layers; beyond either, the multi-head instantiations spill and the wide kernel serves the shape.
constexpr int kMaxHeads = 8;
constexpr int kMaxHeadBytes = 64;

template <typename T, int VECW, int LPR, int VPL, int HV = LPR * VPL, int OP = SDDMM_DOT>
cudaError_t launch_sddmm(Gatv2ScoreParams p, cudaStream_t stream) {
  constexpr int NG = kThreads / LPR;
  // cp.async ring for 16-byte vectors and rows of >= 8 vectors: depth 3 for 256-byte rows, 2 otherwise
  constexpr int PF = (VECW * sizeof(T) == 16 && LPR >= 8) ? (LPR == 16 ? 3 : 2) : 0;
  using SH = SddmmShape<T, VECW, LPR, VPL, PF, HV>;
  // edge-count partition: as segment_reduce (abi.cu choose_config) -- long chunks for large inputs,
  // shorter ones until the grid covers the 148 SMs a few times over
  int chunk = 256;
  while (chunk > LPR && chunk > 8 && (p.E + (int64_t)NG * chunk - 1) / ((int64_t)NG * chunk) < 8 * 148) chunk >>= 1;
  if (chunk < LPR) chunk = LPR;
  p.chunk_edges = chunk;
  const int64_t blocks = (p.E + (int64_t)NG * chunk - 1) / ((int64_t)NG * chunk);
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
  auto launch = [&](auto kern, const auto &params) -> cudaError_t {
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
    kern<<<(unsigned)blocks, kThreads, SH::smem_bytes, stream>>>(params);
    return cudaGetLastError();
  };
  if constexpr (OP == SDDMM_GATV2) return launch(sddmm_coo_kernel<T, VECW, LPR, VPL, PF, HV, OP, Gatv2ScoreParams>, p);
  else return launch(sddmm_coo_kernel<T, VECW, LPR, VPL, PF, HV>, static_cast<const SddmmParams &>(p));
}

template <typename T, int OP>
cudaError_t launch_sddmm_wide(const Gatv2ScoreParams &p, cudaStream_t stream) {
  const int64_t warps_per_block = kThreads / 32;
  const int64_t blocks = (p.E + warps_per_block - 1) / warps_per_block;
  const unsigned grid = (unsigned)(blocks < 148 * 32 ? blocks : 148 * 32);
  if constexpr (OP == SDDMM_GATV2) {
    if (p.H == 1) sddmm_coo_wide_kernel<T, false, OP, Gatv2ScoreParams><<<grid, kThreads, 0, stream>>>(p);
    else sddmm_coo_wide_kernel<T, true, OP, Gatv2ScoreParams><<<grid, kThreads, 0, stream>>>(p);
  } else {
    const SddmmParams &q = p;
    if (p.H == 1) sddmm_coo_wide_kernel<T, false><<<grid, kThreads, 0, stream>>>(q);
    else sddmm_coo_wide_kernel<T, true><<<grid, kThreads, 0, stream>>>(q);
  }
  return cudaGetLastError();
}

// The group shape LPR x VPL fits the row.  H > 1: heads of hv whole 16-byte vectors; the instantiation for HV = hv
// when its results fit the limits above, else the wide kernel.
template <typename T, int OP, int VECW, int LPR, int VPL, int HV = 1>
cudaError_t launch_sddmm_group(const Gatv2ScoreParams &p, int64_t hv, cudaStream_t stream) {
  if (p.H == 1) return launch_sddmm<T, VECW, LPR, VPL, LPR * VPL, OP>(p, stream);
  if constexpr (VECW * sizeof(T) == 16 && HV < LPR * VPL) {
    constexpr int NH = SddmmShape<T, VECW, LPR, VPL, 0, HV>::NH;
    if constexpr (NH <= kMaxHeads && NH * VPL * sizeof(typename AccOf<T>::type) <= kMaxHeadBytes) {
      if (hv == HV) return launch_sddmm<T, VECW, LPR, VPL, HV, OP>(p, stream);
    }
    return launch_sddmm_group<T, OP, VECW, LPR, VPL, HV * 2>(p, hv, stream);
  } else {
    return launch_sddmm_wide<T, OP>(p, stream);
  }
}

template <typename T, int OP, int VECW>
cudaError_t launch_sddmm_shape(const Gatv2ScoreParams &p, int64_t hv, cudaStream_t stream) {
  const int64_t nvec = (p.W + VECW - 1) / VECW;
  if (nvec <= 1) return launch_sddmm_group<T, OP, VECW, 1, 1>(p, hv, stream);
  if (nvec <= 2) return launch_sddmm_group<T, OP, VECW, 2, 1>(p, hv, stream);
  if (nvec <= 4) return launch_sddmm_group<T, OP, VECW, 4, 1>(p, hv, stream);
  if (nvec <= 8) return launch_sddmm_group<T, OP, VECW, 8, 1>(p, hv, stream);
  if (nvec <= 16) return launch_sddmm_group<T, OP, VECW, 16, 1>(p, hv, stream);
  if (nvec <= 32) return launch_sddmm_group<T, OP, VECW, 32, 1>(p, hv, stream);
  if (nvec <= 64) return launch_sddmm_group<T, OP, VECW, 32, 2>(p, hv, stream);
  if constexpr (VECW <= 4) {
    if (nvec <= 128) return launch_sddmm_group<T, OP, VECW, 32, 4>(p, hv, stream);
  }
  return launch_sddmm_wide<T, OP>(p, stream);
}

template <typename T, int OP>
cudaError_t launch_sddmm_type(const Gatv2ScoreParams &p, bool vector_ok, cudaStream_t stream) {
  constexpr int FULL = 16 / (int)sizeof(T);
  if (p.H == 1) {
    if (vector_ok && p.W % FULL == 0) return launch_sddmm_shape<T, OP, FULL>(p, 0, stream);
    return launch_sddmm_shape<T, OP, 1>(p, 0, stream);
  }
  // a head of a power-of-two number of whole 16-byte vectors maps onto lanes; any other goes to the wide kernel
  const int64_t F = p.W / p.H, hv = F / FULL;
  if (vector_ok && F % FULL == 0 && (hv & (hv - 1)) == 0) return launch_sddmm_shape<T, OP, FULL>(p, hv, stream);
  return launch_sddmm_wide<T, OP>(p, stream);
}

}  // namespace

int sddmm(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index, void *out, int64_t E,
          int64_t H, int64_t F, int dtype, int head_major, cudaStream_t stream, const void *att, double slope) {
  Gatv2ScoreParams p;
  p.mat1 = mat1; p.mat2 = mat2; p.row_index = row_index; p.col_index = col_index; p.out = out;
  p.E = E; p.W = H * F; p.H = H; p.head_major = head_major; p.chunk_edges = 0;
  p.att = att; p.slope = slope;
  const bool aligned = ((reinterpret_cast<uintptr_t>(mat1) | reinterpret_cast<uintptr_t>(mat2) |
                         reinterpret_cast<uintptr_t>(att)) & 15) == 0;
  cudaError_t e;
  if (att) {
    switch (dtype) {
      case GEOT_F32: e = launch_sddmm_type<float, SDDMM_GATV2>(p, aligned, stream); break;
      case GEOT_F64: e = launch_sddmm_type<double, SDDMM_GATV2>(p, aligned, stream); break;
      case GEOT_BF16: e = launch_sddmm_type<__nv_bfloat16, SDDMM_GATV2>(p, aligned, stream); break;
      default: e = launch_sddmm_type<__half, SDDMM_GATV2>(p, aligned, stream); break;
    }
  } else {
    switch (dtype) {
      case GEOT_F32: e = launch_sddmm_type<float, SDDMM_DOT>(p, aligned, stream); break;
      case GEOT_F64: e = launch_sddmm_type<double, SDDMM_DOT>(p, aligned, stream); break;
      case GEOT_BF16: e = launch_sddmm_type<__nv_bfloat16, SDDMM_DOT>(p, aligned, stream); break;
      default: e = launch_sddmm_type<__half, SDDMM_DOT>(p, aligned, stream); break;
    }
  }
  if (e != cudaSuccess) return cuda_fail(e, att ? "gatv2_score launch" : H == 1 ? "sddmm_coo launch" : "sddmm_mh launch");
  return GEOT_OK;
}

}  // namespace geot

extern "C" int geot_b200_sddmm_coo(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index,
                                   void *out, int64_t E, int64_t F, int dtype, cudaStream_t stream) {
  if (E < 0 || F <= 0 || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_OK;      // nothing to do (pointers of empty buffers may be null)
  if (!mat1 || !mat2 || !row_index || !col_index || !out) return GEOT_ERR_INVALID_ARG;
  return geot::sddmm(mat1, row_index, mat2, col_index, out, E, 1, F, dtype, 0, stream, nullptr, 0.0);
}

extern "C" int geot_b200_sddmm_mh(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index,
                                  void *out, int64_t E, int64_t H, int64_t F, int dtype, int out_layout,
                                  cudaStream_t stream) {
  if (E < 0 || H <= 0 || F <= 0 || F > INT64_MAX / H || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if (out_layout != GEOT_W_EDGE_HEAD && out_layout != GEOT_W_HEAD_EDGE) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_OK;      // nothing to do (pointers of empty buffers may be null)
  if (!mat1 || !mat2 || !row_index || !col_index || !out) return GEOT_ERR_INVALID_ARG;
  return geot::sddmm(mat1, row_index, mat2, col_index, out, E, H, F, dtype, out_layout == GEOT_W_HEAD_EDGE, stream, nullptr,
                     0.0);
}
