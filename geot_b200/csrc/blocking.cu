// blocking.cu -- src-row blocking of a gather graph for the L2 (format_preprocess family; built once per graph).
//
// Why: a gather op re-reads src rows E / N_src times.  When the src matrix is larger than what the L2 keeps for a
// read-shared working set (measured on B200: ~60 MB of the nominal 126 MB -- profiles/r02a_l2probe.txt: a 59.6 MB src
// is served from L2, a 119 MB one misses 40 % of the time and costs 17 GB of DRAM reads instead of 2.5), the misses
// turn an L2-bound kernel into a DRAM-bound one.  The edge list is therefore regrouped ONCE, stably, by src-row block
// (block b = src rows [b*R, (b+1)*R), R*row_bytes <= ~68 MB): every block is still dst-sorted, and
// geot_b200_segment_reduce_ex reduces block after block -- pass 0 writes every dst row, passes 1.. accumulate
// (segment_reduce.cuh: accumulate, edge_perm) -- so that at any time the gathers touch one block of the matrix.
// Costs 2*(B-1) extra passes over dst and 4 bytes per edge of permutation stream; pays on high-reuse graphs
// (Reddit-shape: degree 492; proteins-shape: 298), not on products-like ones (degree 25): geot_b200_src_blocks_suggest.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cub/device/device_radix_sort.cuh>

#include "internal.h"

namespace {

// key[e] = block of src_index[e]; val[e] = e; per-block edge counts
__global__ void __launch_bounds__(256)
block_keys_kernel(const int64_t *__restrict__ src_index, int64_t E, int64_t rows_per_block, int n_blocks,
                  unsigned char *__restrict__ key, int32_t *__restrict__ val, unsigned long long *__restrict__ counts) {
  __shared__ unsigned int s_cnt[GEOT_MAX_SRC_BLOCKS];
  if (threadIdx.x < GEOT_MAX_SRC_BLOCKS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t b = src_index[e] / rows_per_block;
    b = b < 0 ? 0 : (b >= n_blocks ? n_blocks - 1 : b);
    key[e] = (unsigned char)b;
    val[e] = (int32_t)e;
    atomicAdd(&s_cnt[b], 1u);
  }
  __syncthreads();
  if (threadIdx.x < n_blocks && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

__global__ void __launch_bounds__(256)
regroup_kernel(const int32_t *__restrict__ perm, const int64_t *__restrict__ src_index, const int64_t *__restrict__ dst_index,
               int64_t E, int64_t *__restrict__ src_out, int64_t *__restrict__ dst_out) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int32_t p = perm[e];
    src_out[e] = src_index[p];
    dst_out[e] = dst_index[p];
  }
}

size_t cub_bytes(int64_t E) {
  size_t b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b, (const unsigned char *)nullptr, (unsigned char *)nullptr, (const int32_t *)nullptr,
                                  (int32_t *)nullptr, E, 0, 4);
  return b;
}

}  // namespace

extern "C" {

int geot_b200_src_blocks_suggest(int64_t E, int64_t S, int64_t N_src, int64_t row_bytes) {
  if (E <= 0 || S <= 0 || N_src <= 0 || row_bytes <= 0 || E >= 0x7fffffffLL) return 1;
  // what the L2 keeps of a read-shared matrix (profiles/r02a_l2probe.txt: 59.6 MB stays, 119 MB does not; two blocks
  // of 68 MB measured best on the proteins shape, profiles/r02a_blocks.txt)
  const double kKeep = 68.0 * 1024 * 1024;
  const int64_t kMaxUsefulBlocks = 4;
  const double kMinBlockDegree = 32.0;      // edges per dst row and pass
  const double src_bytes = (double)N_src * (double)row_bytes;
  if (src_bytes <= 64.0 * 1024 * 1024) return 1;             // already resident
  int64_t B = (int64_t)((src_bytes + kKeep - 1) / kKeep);
  // only the measured regime: 2 - 4 blocks (profiles/r02a_blocks_*.json), and passes whose rows stay long.  A pass with a
  // handful of edges per dst row closes a row every few edges and re-reads dst each time: shard 2 of the products shape at
  // 8 GPUs (40 edges per row, a 627 MB src matrix => 9 blocks of 4.5 edges per row) ran 3.2x SLOWER blocked
  // (0.74 vs 0.23 ms, profiles/r02h_n8_bench_n8.json vs r02i shard probe); the byte count below does not see that.
  if (B > kMaxUsefulBlocks) return 1;
  if ((double)E < kMinBlockDegree * (double)B * (double)S) return 1;
  // re-reads avoided (edges whose row would have missed) against the extra passes over dst, with a 2x margin
  const double saved = (double)E * (1.0 - kKeep / src_bytes);
  const double cost = 2.0 * (double)(B - 1) * (double)S;
  return saved > 2.0 * cost ? (int)B : 1;
}

size_t geot_b200_src_blocks_bytes(int64_t E) {
  if (E <= 0) return 256;
  return 2 * align256((size_t)E * 8) + align256((size_t)E * 4);
}

size_t geot_b200_src_blocks_scratch_bytes(int64_t E) {
  if (E <= 0) return 256;
  return 2 * align256((size_t)E) + align256((size_t)E * 4) + align256(GEOT_MAX_SRC_BLOCKS * 8) + align256(cub_bytes(E));
}

int geot_b200_src_blocks_build(const int64_t *src_index, const int64_t *dst_index, int64_t E, int64_t N_src, int n_blocks,
                               void *buf, size_t buf_bytes, void *scratch, size_t scratch_bytes, geot_src_blocks_t *out,
                               cudaStream_t stream) {
  if (!src_index || !dst_index || !buf || !scratch || !out || N_src <= 0) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  if (n_blocks < 1 || n_blocks > GEOT_MAX_SRC_BLOCKS || E >= 0x7fffffffLL) return GEOT_ERR_INVALID_ARG;
  if (buf_bytes < geot_b200_src_blocks_bytes(E) || scratch_bytes < geot_b200_src_blocks_scratch_bytes(E) ||
      ((reinterpret_cast<uintptr_t>(buf) | reinterpret_cast<uintptr_t>(scratch)) & 255))
    return GEOT_ERR_WORKSPACE;
  char *p = static_cast<char *>(buf);
  int64_t *dst_b = reinterpret_cast<int64_t *>(p); p += align256((size_t)E * 8);
  int64_t *src_b = reinterpret_cast<int64_t *>(p); p += align256((size_t)E * 8);
  int32_t *perm = reinterpret_cast<int32_t *>(p);
  char *q = static_cast<char *>(scratch);
  unsigned char *key_in = reinterpret_cast<unsigned char *>(q); q += align256((size_t)E);
  unsigned char *key_out = reinterpret_cast<unsigned char *>(q); q += align256((size_t)E);
  int32_t *val_in = reinterpret_cast<int32_t *>(q); q += align256((size_t)E * 4);
  unsigned long long *counts = reinterpret_cast<unsigned long long *>(q); q += align256(GEOT_MAX_SRC_BLOCKS * 8);
  void *cub_tmp = q;
  size_t cb = cub_bytes(E);
  const int64_t rows_per_block = (N_src + n_blocks - 1) / n_blocks;
  CUDA_TRY(cudaMemsetAsync(counts, 0, GEOT_MAX_SRC_BLOCKS * 8, stream));
  const unsigned nb = (unsigned)std::min<int64_t>((E + 255) / 256, 148 * 16);
  block_keys_kernel<<<nb, 256, 0, stream>>>(src_index, E, rows_per_block, n_blocks, key_in, val_in, counts);
  CUDA_TRY(cudaGetLastError());
  int bits = 1;
  while ((1 << bits) < n_blocks) ++bits;
  // LSD radix sort on the block id: stable, so every block keeps the (dst, src) order of the caller's list
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, key_in, key_out, val_in, perm, E, 0, bits, stream));
  regroup_kernel<<<nb, 256, 0, stream>>>(perm, src_index, dst_index, E, src_b, dst_b);
  CUDA_TRY(cudaGetLastError());
  unsigned long long h[GEOT_MAX_SRC_BLOCKS];
  CUDA_TRY(cudaMemcpyAsync(h, counts, sizeof(h), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  out->E = E;
  out->n_blocks = n_blocks;
  out->reserved = 0;
  out->bounds[0] = 0;
  for (int b = 0; b < GEOT_MAX_SRC_BLOCKS; ++b) out->bounds[b + 1] = out->bounds[b] + (b < n_blocks ? (int64_t)h[b] : 0);
  if (out->bounds[n_blocks] != E) return GEOT_ERR_INVALID_ARG;
  out->dst_index = dst_b;
  out->src_index = src_b;
  out->edge_perm = perm;
  return GEOT_OK;
}

}  // extern "C"
