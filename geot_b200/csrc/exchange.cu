// exchange.cu -- device helpers of the multi-GPU path (geot_b200/dist.py; SURVEY.md 8e).  New functionality:
// the reference has no distributed code.
//
// The dst-sharded gather ops overlap the exchange of the src rows with the reduction: a rank's edges are split once
// per graph into a src-local and a src-remote bucket (stable, so both stay dst-sorted); the local bucket is reduced
// while the remote rows travel, the remote bucket afterwards with accumulate (segment_reduce.cuh).  Here:
// push_rows (the fused pack + transfer over peer memory of the "push" transport) and permute_edges (per-head
// weights into bucket order; one weight per edge needs no pass: the kernel reads weight[edge_perm[e]]).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "internal.h"

namespace {

// out[e*words + k] = in[perm[e]*words + k]: edge operands (weights) into bucket order, 4-byte words
__global__ void __launch_bounds__(256)
permute_edges_kernel(const uint32_t *__restrict__ in, const int64_t *__restrict__ perm, uint32_t *__restrict__ out,
                     int64_t E, int words) {
  const int64_t n = E * words;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i / words;
    const int k = (int)(i - e * words);
    out[i] = in[perm[e] * words + k];
  }
}
__global__ void __launch_bounds__(256)
permute_edges16_kernel(const uint16_t *__restrict__ in, const int64_t *__restrict__ perm, uint16_t *__restrict__ out,
                       int64_t E, int halves) {
  const int64_t n = E * halves;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i / halves;
    const int k = (int)(i - e * halves);
    out[i] = in[perm[e] * halves + k];
  }
}

// 16-byte pieces: packs whole feature rows (the rows a peer asked for) at full vector width
__global__ void __launch_bounds__(256)
permute_rows16_kernel(const uint4 *__restrict__ in, const int64_t *__restrict__ perm, uint4 *__restrict__ out, int64_t E,
                      int vecs) {
  const int64_t n = E * vecs;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i / vecs;
    const int k = (int)(i - e * vecs);
    out[i] = in[perm[e] * vecs + k];
  }
}

// Fused pack + transfer over peer memory: row e of the send list goes straight into the receive buffer of the
// GPU that asked for it -- bases[dest_peer[e]] is that GPU's buffer mapped into this process (NVLink P2P stores,
// 16-byte vectors), dest_row[e] the row slot the receiver's src ids point at.  No staging buffer, no NCCL call.
//
// The transfer is NVLink-bound (660 GB/s per direction measured at N = 4, profiles/r02j_n4_timeline.txt) and runs
// BESIDE the reduction of the src-local edge bucket, so the kernel is built to leave the SMs to that reduction: a small
// persistent grid (max_ctas, the caller's choice: geot_b200_push_rows_ex; CTAs of 128 threads, <= 48 registers: they fit
// next to the resident CTAs of segment_reduce_kernel) in which every thread keeps kPushUnroll 16-byte pieces in flight (2 CTAs per SM: 148 x 2 x 128 x 4 x
// 16 B = 2.4 MB, several times the link's bandwidth-delay product).  Round 2's first version launched 4736 CTAs of 256 threads
// with one piece in flight per thread: alone it reached the same rate, but next to the reduction the two kernels took
// turns on the SMs (local bucket 0.24 ms + push 0.14 ms = the 0.13 ms that the N = 4 step lost against its parts).
constexpr int kPushThreads = 128;
constexpr int kPushUnroll = 4;

template <typename V>
__global__ void __launch_bounds__(kPushThreads, 10)
push_rows_kernel(const V *__restrict__ x, const int64_t *__restrict__ rows, const int32_t *__restrict__ dest_peer,
                 const int64_t *__restrict__ dest_row, V *const *__restrict__ bases, int64_t n, int vecs, int vecs_shift) {
  const int64_t total = n * vecs;
  const int64_t stride = (int64_t)gridDim.x * kPushThreads;
  for (int64_t i0 = (int64_t)blockIdx.x * kPushThreads + threadIdx.x; i0 < total; i0 += stride * kPushUnroll) {
    V v[kPushUnroll];
    V *q[kPushUnroll];
#pragma unroll
    for (int u = 0; u < kPushUnroll; ++u) {
      const int64_t i = i0 + u * stride;
      q[u] = nullptr;
      if (i < total) {
        const int64_t e = vecs_shift >= 0 ? (i >> vecs_shift) : (i / vecs);
        const int64_t k = i - e * vecs;
        v[u] = x[rows[e] * vecs + k];
        q[u] = bases[dest_peer[e]] + (dest_row[e] * vecs + k);
      }
    }
#pragma unroll
    for (int u = 0; u < kPushUnroll; ++u)
      if (q[u] != nullptr) *q[u] = v[u];
  }
}

}  // namespace

extern "C" {

int geot_b200_permute_edges(const void *in, const int64_t *perm, void *out, int64_t E, int64_t bytes_per_edge,
                            cudaStream_t stream) {
  if (E < 0 || bytes_per_edge <= 0 || (bytes_per_edge & 1)) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_OK;       // nothing to move (an empty tensor's pointer may be null)
  if (!in || !perm || !out) return GEOT_ERR_INVALID_ARG;
  // widest move that both the record size and the base pointers allow (a view may start mid-vector)
  const uintptr_t addr = reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out);
  if (addr & 1) return GEOT_ERR_INVALID_ARG;
  const bool vec16 = bytes_per_edge % 16 == 0 && (addr & 15) == 0;
  const bool vec4 = bytes_per_edge % 4 == 0 && (addr & 3) == 0;
  const int64_t n = E * (vec16 ? bytes_per_edge / 16 : (vec4 ? bytes_per_edge / 4 : bytes_per_edge / 2));
  const unsigned blocks = (unsigned)((n + 255) / 256 < 148 * 32 ? (n + 255) / 256 : 148 * 32);
  if (vec16)
    permute_rows16_kernel<<<blocks, 256, 0, stream>>>(static_cast<const uint4 *>(in), perm, static_cast<uint4 *>(out), E,
                                                      (int)(bytes_per_edge / 16));
  else if (vec4)
    permute_edges_kernel<<<blocks, 256, 0, stream>>>(static_cast<const uint32_t *>(in), perm, static_cast<uint32_t *>(out), E,
                                                     (int)(bytes_per_edge / 4));
  else
    permute_edges16_kernel<<<blocks, 256, 0, stream>>>(static_cast<const uint16_t *>(in), perm, static_cast<uint16_t *>(out),
                                                       E, (int)(bytes_per_edge / 2));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "permute_edges_kernel");
  return GEOT_OK;
}

int geot_b200_push_rows(const void *x, const int64_t *rows, const int32_t *dest_peer, const int64_t *dest_row,
                        void *const *peer_bases, int64_t n, int64_t row_bytes, int peers_aligned16, cudaStream_t stream) {
  return geot_b200_push_rows_ex(x, rows, dest_peer, dest_row, peer_bases, n, row_bytes, peers_aligned16, 0, stream);
}

int geot_b200_push_rows_ex(const void *x, const int64_t *rows, const int32_t *dest_peer, const int64_t *dest_row,
                           void *const *peer_bases, int64_t n, int64_t row_bytes, int peers_aligned16, int max_ctas,
                           cudaStream_t stream) {
  if (n < 0 || row_bytes <= 0 || (row_bytes & 1)) return GEOT_ERR_INVALID_ARG;
  if (n == 0) return GEOT_OK;
  if (!x || !rows || !dest_peer || !dest_row || !peer_bases) return GEOT_ERR_INVALID_ARG;
  if (reinterpret_cast<uintptr_t>(x) & 1) return GEOT_ERR_INVALID_ARG;
  // the peer bases live in device memory: the caller vouches for their alignment (symmetric allocations are)
  const bool vec16 = row_bytes % 16 == 0 && peers_aligned16 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  const bool vec4 = row_bytes % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 3) == 0;      // (bases: >= 4-byte aligned rows)
  const int64_t vecs = vec16 ? row_bytes / 16 : (vec4 ? row_bytes / 4 : row_bytes / 2);
  const int64_t total = n * vecs;
  int shift = -1;
  if ((vecs & (vecs - 1)) == 0) { shift = 0; while ((1LL << shift) < vecs) ++shift; }
  // max_ctas > 0: a small persistent grid that leaves the SMs to a concurrent reduction (see push_rows_kernel);
  // 0: the transfer has the GPU to itself.  GEOT_B200_PUSH_CTAS overrides a positive max_ctas (tuning).
  int64_t want = max_ctas > 0 ? max_ctas : 148LL * 10;
  if (max_ctas > 0) { if (const char *s = getenv("GEOT_B200_PUSH_CTAS")) { if (atoi(s) > 0) want = atoi(s); } }
  const int64_t need = (total + (int64_t)kPushThreads * kPushUnroll - 1) / ((int64_t)kPushThreads * kPushUnroll);
  const unsigned blocks = (unsigned)(need < want ? need : want);
  if (vec16)
    push_rows_kernel<uint4><<<blocks, kPushThreads, 0, stream>>>(static_cast<const uint4 *>(x), rows, dest_peer, dest_row,
                                                                 reinterpret_cast<uint4 *const *>(peer_bases), n, (int)vecs, shift);
  else if (vec4)
    push_rows_kernel<uint32_t><<<blocks, kPushThreads, 0, stream>>>(static_cast<const uint32_t *>(x), rows, dest_peer, dest_row,
                                                                    reinterpret_cast<uint32_t *const *>(peer_bases), n, (int)vecs,
                                                                    shift);
  else      // bf16 / fp16 rows with an odd element count
    push_rows_kernel<uint16_t><<<blocks, kPushThreads, 0, stream>>>(static_cast<const uint16_t *>(x), rows, dest_peer, dest_row,
                                                                    reinterpret_cast<uint16_t *const *>(peer_bases), n, (int)vecs,
                                                                    shift);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "push_rows_kernel");
  return GEOT_OK;
}

}  // extern "C"
