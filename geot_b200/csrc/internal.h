// internal.h -- shared by the translation units of libgeot_b200.so and not installed.  The library is compiled with
// -fvisibility=hidden, so nothing declared here is exported: the dynamic symbols are the geot_b200_* functions of
// include/geot_b200.h only.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/geot_b200.h"

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
inline size_t dtype_size(int dt) { return dt == GEOT_F64 ? 8 : (dt == GEOT_F32 ? 4 : 2); }

inline int env_int(const char *name, int dflt) {
  const char *s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// Records "what: <CUDA error text>" for geot_b200_last_cuda_error() on this thread; returns GEOT_ERR_CUDA (abi.cu).
int cuda_fail(cudaError_t e, const char *what);

#define CUDA_TRY(expr)                                    \
  do {                                                    \
    cudaError_t e__ = (expr);                             \
    if (e__ != cudaSuccess) return cuda_fail(e__, #expr); \
  } while (0)

// What the public entries do not expose: how empty rows are cleared and which rows the call owns.
struct Extra {
  int clear_mode = 0;          // 0: rows without edges are zeroed by this call; 1: the caller owns that (never clear)
  int64_t fill_lo = 0;         // rows [fill_lo, fill_hi) belong to this call (host-entry slices); fill_hi < 0: [0, S)
  int64_t fill_hi = -1;
};

// The device entry behind geot_b200_segment_reduce{,_ex} and every slice of the host-buffer entries (abi.cu).
int segment_reduce_impl(const void *src, const int64_t *src_index, const int64_t *dst_index,
                        const void *weight, void *dst, int64_t E, int64_t S, int64_t H, int64_t F,
                        int dtype, int reduce, int weight_layout, int sorted, const geot_plan_t *plan,
                        void *workspace, size_t workspace_bytes, cudaStream_t stream, const geot_reduce_opts_t *opts,
                        const Extra &ex);

// The SDDMM launcher (sddmm.cu): out[e, h] = sum over a head's columns of mat1[row_index[e]] * mat2[col_index[e]], or
// with att != null the GATv2 score att * leaky_relu(mat1 + mat2) of slope `slope`.  Arguments already validated.
namespace geot {
int sddmm(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index, void *out, int64_t E,
          int64_t H, int64_t F, int dtype, int head_major, cudaStream_t stream, const void *att, double slope);
}  // namespace geot
