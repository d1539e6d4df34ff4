// abi.cu -- the extern "C" boundary declared in include/geot_b200.h for device buffers: argument checking, kernel
// shape selection (replaces the reference's decision trees, csrc/cuda/wrapper/*_rule.h) and format_preprocess.  The
// host-buffer entries are in host.cu.  No torch / ATen types here; the torch bindings (bindings.cpp) and any other
// host (ctypes, cgo, JNI) call these functions.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>

#include "internal.h"
#include "kernels/launch.h"

static thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e, const char *what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
  return GEOT_ERR_CUDA;
}

namespace {

inline size_t acc_size(int dt) { return dt == GEOT_F64 ? 8 : 4; }
inline int pow2ceil(int64_t x) { int p = 1; while (p < x) p <<= 1; return p; }

// ---- kernel shape + edge partition --------------------------------------------------------------
struct Config {
  geot::Shape shape;
  int chunk_edges;
  int64_t tile_edges;
  int64_t n_tiles;
};

// `vector_ok`: rows are 16-byte addressable (per-head width multiple of the vector width and
// 16-byte aligned base pointers); otherwise the element-wise kernels are used.
Config choose_config(int64_t E, int64_t W, int64_t F, int dtype, bool vector_ok, bool gather = true) {
  Config c;
  const int full = (int)(16 / dtype_size(dtype));
  const int vecw = (vector_ok && F % full == 0) ? full : 1;
  const int64_t nvec = (W + vecw - 1) / vecw;
  int lpr, vpl;
  if (nvec <= 32) {
    lpr = pow2ceil(nvec);
    vpl = 1;
  } else {
    // wider rows: several vectors per lane, capped so that the accumulators stay within 16 registers
    // (fp32: 4 vectors, fp64: 4, bf16/fp16 with 8-element vectors: 2); beyond that, column tiles
    const int vpl_max = (vecw == 8) ? 2 : 4;
    lpr = 32;
    vpl = (nvec <= 64 || vpl_max == 2) ? 2 : 4;
  }
  c.shape.vecw = vecw;
  c.shape.lpr = lpr;
  c.shape.vpl = vpl;
  c.shape.col_tiles = (int)((nvec + (int64_t)lpr * vpl - 1) / ((int64_t)lpr * vpl));
  c.shape.wm = 0;
  // gathered rows through the cp.async shared-memory ring for the kernels that have one (sum, 16-byte vectors, rows
  // of >= 8 vectors).  Default: the lean ring, depth 3 (4 stages of 2 KB per warp = 6 KB in flight per warp); depth 7
  // where the rows are a pure DRAM stream (index_scatter: src row = edge id) -- profiles/r01c_ring_ab.txt.  The
  // launcher falls back to the first-generation ring where the lean ring does not apply (fp64, per-head weights).
  // GEOT_B200_RING=0 selects the register path, 2 / 3 the first-generation ring, 32 + depth a lean depth.
  c.shape.pf = env_int("GEOT_B200_RING", (vecw > 1 && lpr >= 8) ? (geot::kLeanFlag | (gather ? 3 : 7)) : 0);
  const int ng = geot::kThreads / lpr;
  // Edge-count partition: every group owns `chunk` consecutive edges.  Longer chunks amortise the
  // per-chunk carry handling; shorter ones keep small inputs spread over all 148 SMs.
  int chunk = env_int("GEOT_B200_CHUNK", 0);
  if (chunk <= 0) {
    chunk = 256;
    // at least 3.5 tiles per SM (measured on the two small BASELINE shapes, profiles/r02a_chunk_sweep_small.txt and
    // r02s_tune.txt: config #1 index_scatter 0.064 ms at chunk 128 = 489 tiles -> 0.057 at 64 = 977; arxiv mh_spmm 0.128 at
    // 128 = 1139 tiles -> 0.116 at 256 = 570)
    while (chunk > 8 && (E + (int64_t)ng * chunk - 1) / ((int64_t)ng * chunk) < 518) chunk >>= 1;
  }
  // (Sizing the grid in whole waves of resident CTAs -- shrinking the chunk until the tiles fill an integer number of
  // waves -- was measured on the shapes that are only a few waves deep and changed nothing: config #1 0.065 / 0.066 ms,
  // arxiv mh_spmm 0.138 / 0.138, the 8 products-shape shards 0.220-0.262 / 0.221-0.257, profiles/r02l_tune.txt,
  // r02l_shard_probe.txt.  The tiles are short enough for the block scheduler to even out the last wave.  Removed.)
  c.chunk_edges = chunk;
  c.tile_edges = (int64_t)ng * chunk;
  c.n_tiles = (E + c.tile_edges - 1) / c.tile_edges;
  return c;
}

struct Workspace {
  void *carry_head, *carry_tail;
  long long *head_cnt, *tail_cnt;
  int64_t *tail_row;
  unsigned char *flags;
  size_t bytes;
};

Workspace carve(void *base, int64_t n_tiles, int64_t W, int dtype) {
  Workspace w;
  char *p = static_cast<char *>(base);
  size_t off = 0;
  const size_t carry = align256((size_t)n_tiles * (size_t)W * acc_size(dtype));
  w.carry_head = p + off; off += carry;
  w.carry_tail = p + off; off += carry;
  w.head_cnt = reinterpret_cast<long long *>(p + off); off += align256((size_t)n_tiles * 8);
  w.tail_cnt = reinterpret_cast<long long *>(p + off); off += align256((size_t)n_tiles * 8);
  w.tail_row = reinterpret_cast<int64_t *>(p + off); off += align256((size_t)n_tiles * 8);
  w.flags = reinterpret_cast<unsigned char *>(p + off); off += align256((size_t)n_tiles + 1);
  w.bytes = off;
  return w;
}

geot::launch_fn pick_launcher(int dtype, int reduce) {
  using namespace geot;
  const int r = (reduce == GEOT_MEAN) ? GEOT_SUM : reduce;
#ifdef GEOT_MINIMAL   // tuning builds carry the fp32 sum kernels only
  return (dtype == GEOT_F32 && r == 0) ? launch_f32_0 : nullptr;
#else
#define ROW(TN) \
  switch (r) { case 0: return launch_##TN##_0; case 2: return launch_##TN##_2; \
               case 3: return launch_##TN##_3; case 4: return launch_##TN##_4; } break;
  switch (dtype) {
    case GEOT_F32: ROW(f32)
    case GEOT_F64: ROW(f64)
    case GEOT_BF16: ROW(bf16)
    case GEOT_F16: ROW(f16)
  }
#undef ROW
  return nullptr;
#endif
}

// ---- format_preprocess kernels --------------------------------------------------------------------
struct PlanStats {
  long long num_segments;
  long long max_degree;
  long long max_row;
  int unsorted;
  int pad;
};

// rowptr[r] = first edge position with dst_index >= r  (lower bound; r = 0..S)
__global__ void rowptr_kernel(const int64_t *__restrict__ idx, int64_t E, int64_t S, int64_t *__restrict__ rowptr) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > S) return;
  int64_t lo = 0, hi = E;
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (idx[mid] < r) lo = mid + 1; else hi = mid;
  }
  rowptr[r] = lo;
}

__global__ void index_stats_kernel(const int64_t *__restrict__ idx, int64_t E, PlanStats *stats) {
  long long heads = 0, mx = 0;
  int unsorted = 0;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = idx[e];
    mx = max(mx, (long long)b);
    if (e == 0) { heads += 1; continue; }
    const int64_t a = idx[e - 1];
    heads += (a != b);
    unsorted |= (b < a);
  }
  for (int o = 16; o > 0; o >>= 1) {
    heads += __shfl_xor_sync(0xffffffffu, heads, o);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    unsorted |= __shfl_xor_sync(0xffffffffu, unsorted, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (heads) atomicAdd(reinterpret_cast<unsigned long long *>(&stats->num_segments), (unsigned long long)heads);
    if (mx) atomicMax(&stats->max_row, mx);
    if (unsorted) atomicOr(&stats->unsorted, 1);
  }
}

__global__ void degree_stats_kernel(const int64_t *__restrict__ rowptr, int64_t S, PlanStats *stats) {
  long long m = 0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S; r += (int64_t)gridDim.x * blockDim.x)
    m = max(m, (long long)(rowptr[r + 1] - rowptr[r]));
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(&stats->max_degree, m);
}

// shard g starts at the segment boundary nearest to g*E/parts
__global__ void shard_kernel(const int64_t *__restrict__ rowptr, int64_t S, int64_t E, int parts,
                             int64_t *row_bounds, int64_t *edge_bounds) {
  const int g = threadIdx.x;
  if (g > parts) return;
  if (g == 0) { row_bounds[0] = 0; edge_bounds[0] = 0; return; }
  if (g == parts) { row_bounds[g] = S; edge_bounds[g] = E; return; }
  const int64_t target = (E / parts) * g + ((E % parts) * g) / parts;
  int64_t lo = 0, hi = S;  // first r with rowptr[r] >= target
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (rowptr[mid] < target) lo = mid + 1; else hi = mid;
  }
  int64_t r = lo;
  if (r > 0 && target - rowptr[r - 1] < rowptr[r] - target) r -= 1;
  row_bounds[g] = r;
  edge_bounds[g] = rowptr[r];
}

__global__ void iota_kernel(int64_t *p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}
__global__ void gather_index_kernel(const int64_t *__restrict__ perm, const int64_t *__restrict__ in, int64_t *out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[perm[i]];
}

// Rows that receive no edge must read 0.  With a plan the empty rows are known (rowptr[r+1] == rowptr[r], and every row
// at or beyond the plan's S): a warp checks 32 rows, then zero-fills the empty ones cooperatively -- the writes are the
// empty rows only, not a memset of the whole dst, and the main kernel runs its plain instantiation.  (Zero-filling inside
// the main kernel -- the group that sees the jump in the sorted index fills the gap -- is what a call WITHOUT a plan does;
// on the products shape with a quarter of the rows isolated it costs 0.18 ms of the step against 0.04 ms here,
// profiles/r02y_tune_gaps.txt.)
__global__ void __launch_bounds__(256)
zero_empty_rows_kernel(const int64_t *__restrict__ rowptr, int64_t plan_rows, int64_t S, int64_t row_bytes, char *dst, int vec16) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp * 32; base < S; base += n_warps * 32) {
    const int64_t r = base + lane;
    bool empty = false;
    if (r < S) empty = (r >= plan_rows) || (rowptr[r + 1] == rowptr[r]);
    unsigned m = __ballot_sync(0xffffffffu, empty);
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      char *row = dst + (base + b) * row_bytes;
      if (vec16) {
        for (int64_t o = (int64_t)lane * 16; o < row_bytes; o += 32 * 16) *reinterpret_cast<uint4 *>(row + o) = make_uint4(0, 0, 0, 0);
      } else {
        for (int64_t o = (int64_t)lane * 2; o < row_bytes; o += 32 * 2) *reinterpret_cast<unsigned short *>(row + o) = 0;
      }
    }
  }
}

// ---- index_scatter(sorted = False), sum, fp32: 128-bit vector atomics ------------------------------------------------
// The reference's unsorted kernel (scatter_reduce_kernel, csrc/cuda/index_scatter_kernel.cuh:204-263) issues one scalar
// atomicAdd per element after a torch::zeros.  Here every thread streams 16 bytes of src (read once: evict-first) and
// adds them with ONE red.global.add.v4.f32 (REDG.E.ADD.F32x4, sm_90+): a quarter of the atomic operations, the dst
// rows stay in L2.  Like the reference's, the summation order is the hardware's: not bit-reproducible run to run
// (geot_b200_set_unsorted_mode(1) selects the deterministic sort-based path instead; it is what every other dtype and
// reduce op uses).  Measured beside the reference kernel by scripts/compare_reference_cuda.py unsorted.
__device__ __forceinline__ void red_add(float *q, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void red_add(float *q, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(q), "f"(v) : "memory");
}
__device__ __forceinline__ float4 ld_once(const float4 *p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float ld_once(const float *p, uint64_t pol) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
constexpr int kScatterUnroll = 4;
// V = float4 (rows of whole 16-byte pieces) or float; `pieces` = pieces per row, shift = log2(pieces) or -1
template <typename V>
__global__ void __launch_bounds__(256)
scatter_add_kernel(const V *__restrict__ src, const int64_t *__restrict__ src_index, const int64_t *__restrict__ index,
                   float *__restrict__ dst, int64_t E, int pieces, int shift, int64_t S) {
  constexpr int PW = (int)(sizeof(V) / sizeof(float));
  const int64_t total = E * pieces;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const uint64_t pol = geot::policy_evict_first();
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += stride * kScatterUnroll) {
    V v[kScatterUnroll];
    float *q[kScatterUnroll];
#pragma unroll
    for (int u = 0; u < kScatterUnroll; ++u) {
      const int64_t i = i0 + u * stride;
      q[u] = nullptr;
      if (i < total) {
        const int64_t e = shift >= 0 ? (i >> shift) : (i / pieces);
        const int64_t k = i - e * pieces;
        const int64_t row = index[e];
        const int64_t srow = src_index ? src_index[e] : e;
        v[u] = ld_once(src + srow * pieces + k, pol);
        if (row >= 0 && row < S) q[u] = dst + (row * pieces + k) * PW;    // (an index outside [0, S) is dropped, not written)
      }
    }
#pragma unroll
    for (int u = 0; u < kScatterUnroll; ++u)
      if (q[u] != nullptr) red_add(q[u], v[u]);
  }
}

int g_unsorted_mode = 0;      // 0: vector atomics where they apply (fp32 sum); 1: always the deterministic sort path

// CSR row pointer -> COO row index: one thread per edge, binary search of the edge position in rowptr
// (upper bound - 1).  Rows are found independently, so the kernel is a single coalesced write pass.
template <typename P>
__global__ void csr_rows_kernel(const P *__restrict__ rowptr, int64_t S, int64_t E, int64_t *__restrict__ row) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t lo = 0, hi = S;   // last r with rowptr[r] <= e
  while (hi - lo > 1) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if ((int64_t)rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  row[e] = lo;
}

// ---- instrumentation: event pairs around the main kernel ------------------------------------------
struct Profile {
  int n = 0;
  long long calls = 0;
  cudaEvent_t *start = nullptr, *stop = nullptr;
};
thread_local Profile g_prof;

constexpr int kMaxParts = 64;
size_t plan_tail_bytes() { return align256(sizeof(PlanStats)) + align256(2 * (kMaxParts + 1) * sizeof(int64_t)); }

int bits_for(int64_t S) { int b = 1; while (b < 63 && ((int64_t)1 << b) < S) ++b; return b; }

}  // namespace

// ==================================================================================================
extern "C" {

int geot_b200_version(void) { return GEOT_B200_VERSION; }
int geot_b200_arch(void) { return 100; }

const char *geot_b200_status_string(int s) {
  switch (s) {
    case GEOT_OK: return "ok";
    case GEOT_ERR_INVALID_ARG: return "invalid argument";
    case GEOT_ERR_UNSUPPORTED: return "unsupported";
    case GEOT_ERR_WORKSPACE: return "workspace too small or misaligned";
    case GEOT_ERR_CUDA: return "CUDA error";
    case GEOT_ERR_EMPTY: return "empty index";
  }
  return "unknown status";
}
const char *geot_b200_last_cuda_error(void) { return g_cuda_err; }

int geot_b200_index_last(const int64_t *dst_index, int64_t E, int64_t *last, cudaStream_t stream) {
  if (!dst_index || !last) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  CUDA_TRY(cudaMemcpyAsync(last, dst_index + (E - 1), sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  return GEOT_OK;
}

size_t geot_b200_plan_bytes(int64_t E, int64_t S) {
  (void)E;
  if (S < 0) return 0;
  return align256((size_t)(S + 1) * sizeof(int64_t)) + plan_tail_bytes();
}

int geot_b200_format_preprocess(const int64_t *dst_index, int64_t E, int64_t S, void *plan_buf,
                                size_t plan_bytes, geot_plan_t *plan, cudaStream_t stream) {
  if (!dst_index || !plan_buf || !plan || S <= 0) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  if (plan_bytes < geot_b200_plan_bytes(E, S) || (reinterpret_cast<uintptr_t>(plan_buf) & 255)) return GEOT_ERR_WORKSPACE;
  int64_t *rowptr = static_cast<int64_t *>(plan_buf);
  PlanStats *stats = reinterpret_cast<PlanStats *>(static_cast<char *>(plan_buf) + align256((size_t)(S + 1) * 8));
  CUDA_TRY(cudaMemsetAsync(stats, 0, sizeof(PlanStats), stream));
  const int thr = 256;
  rowptr_kernel<<<(unsigned)((S + 1 + thr - 1) / thr), thr, 0, stream>>>(dst_index, E, S, rowptr);
  CUDA_TRY(cudaGetLastError());
  const unsigned nb = (unsigned)std::min<int64_t>((E + thr - 1) / thr, 148 * 16);
  index_stats_kernel<<<nb, thr, 0, stream>>>(dst_index, E, stats);
  CUDA_TRY(cudaGetLastError());
  const unsigned nb2 = (unsigned)std::min<int64_t>((S + thr - 1) / thr, 148 * 16);
  degree_stats_kernel<<<nb2, thr, 0, stream>>>(rowptr, S, stats);
  CUDA_TRY(cudaGetLastError());
  PlanStats h;
  CUDA_TRY(cudaMemcpyAsync(&h, stats, sizeof(h), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  plan->E = E;
  plan->S = S;
  plan->num_segments = h.num_segments;
  plan->max_degree = h.max_degree;
  plan->is_sorted = h.unsorted ? 0 : 1;
  plan->has_gaps = (h.unsorted || h.num_segments < S) ? 1 : 0;
  plan->rowptr = rowptr;
  plan->max_row = h.max_row;
  return GEOT_OK;
}

int geot_b200_plan_shards(const geot_plan_t *plan, int parts, int64_t *row_bounds, int64_t *edge_bounds,
                          cudaStream_t stream) {
  if (!plan || !plan->rowptr || !row_bounds || !edge_bounds || parts < 1 || parts > kMaxParts) return GEOT_ERR_INVALID_ARG;
  char *base = reinterpret_cast<char *>(const_cast<int64_t *>(plan->rowptr));
  int64_t *d_bounds = reinterpret_cast<int64_t *>(base + align256((size_t)(plan->S + 1) * 8) + align256(sizeof(PlanStats)));
  shard_kernel<<<1, kMaxParts + 1, 0, stream>>>(plan->rowptr, plan->S, plan->E, parts, d_bounds, d_bounds + (kMaxParts + 1));
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(row_bounds, d_bounds, (parts + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaMemcpyAsync(edge_bounds, d_bounds + (kMaxParts + 1), (parts + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  CUDA_TRY(cudaStreamSynchronize(stream));
  return GEOT_OK;
}

int geot_b200_csr_to_coo(const void *rowptr, int rowptr_bits, int64_t S, int64_t E, int64_t *row_index,
                         cudaStream_t stream) {
  if (!rowptr || !row_index || S <= 0 || E < 0 || (rowptr_bits != 32 && rowptr_bits != 64)) return GEOT_ERR_INVALID_ARG;
  if (E == 0) return GEOT_OK;
  const unsigned nb = (unsigned)((E + 255) / 256);
  if (rowptr_bits == 64) csr_rows_kernel<int64_t><<<nb, 256, 0, stream>>>(static_cast<const int64_t *>(rowptr), S, E, row_index);
  else csr_rows_kernel<int32_t><<<nb, 256, 0, stream>>>(static_cast<const int32_t *>(rowptr), S, E, row_index);
  CUDA_TRY(cudaGetLastError());
  return GEOT_OK;
}

size_t geot_b200_workspace_bytes(int64_t E, int64_t W, int dtype, int sorted) {
  if (E <= 0 || W <= 0) return 256;
  // the vector and the element-wise shapes partition differently: size for the larger
  size_t best = 0;
  for (int v = 0; v < 2; ++v) {
    const Config c = choose_config(E, W, W, dtype, v == 1);
    Workspace w = carve(nullptr, c.n_tiles, W, dtype);
    best = std::max(best, w.bytes);
  }
  if (sorted) return best;
  // sorted == 0 additionally needs the sort buffers (keys, permutation, cub scratch)
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int64_t *)nullptr, (int64_t *)nullptr,
                                  (const int64_t *)nullptr, (int64_t *)nullptr, E);
  return best + 4 * align256((size_t)E * 8) + align256(cub_bytes);
}

}  // extern "C"

int segment_reduce_impl(const void *src, const int64_t *src_index, const int64_t *dst_index,
                        const void *weight, void *dst, int64_t E, int64_t S, int64_t H, int64_t F,
                        int dtype, int reduce, int weight_layout, int sorted, const geot_plan_t *plan,
                        void *workspace, size_t workspace_bytes, cudaStream_t stream, const geot_reduce_opts_t *opts,
                        const Extra &ex) {
  if (!src || !dst_index || !dst) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  if (S <= 0 || H <= 0 || F <= 0) return GEOT_ERR_INVALID_ARG;
  if (dtype < GEOT_F32 || dtype > GEOT_F16 || reduce < GEOT_SUM || reduce > GEOT_PROD) return GEOT_ERR_INVALID_ARG;
  if (weight_layout < GEOT_W_NONE || weight_layout > GEOT_W_HEAD_EDGE) return GEOT_ERR_INVALID_ARG;
  if ((weight_layout == GEOT_W_NONE) != (weight == nullptr)) return GEOT_ERR_INVALID_ARG;
  if (weight_layout == GEOT_W_EDGE && H != 1) return GEOT_ERR_INVALID_ARG;
  if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return GEOT_ERR_WORKSPACE;
  if (plan && (plan->E != E || plan->S > S)) return GEOT_ERR_INVALID_ARG;
  const bool accumulate = opts && opts->accumulate;
  const int32_t *edge_perm = opts ? opts->edge_perm : nullptr;
  const int64_t *mean_rowptr = opts ? opts->mean_rowptr : nullptr;
  if (opts && opts->struct_size != sizeof(geot_reduce_opts_t)) return GEOT_ERR_INVALID_ARG;
  // bucketed passes add partial SUMS (mean: each already divided by the row's full degree)
  if (accumulate && reduce != GEOT_SUM && !(reduce == GEOT_MEAN && mean_rowptr)) return GEOT_ERR_UNSUPPORTED;
  if (edge_perm && (weight_layout != GEOT_W_EDGE || (reduce != GEOT_SUM && reduce != GEOT_MEAN) || !sorted)) return GEOT_ERR_UNSUPPORTED;
  const int64_t W = H * F;
  geot::launch_fn launch = pick_launcher(dtype, reduce);
  if (!launch) return GEOT_ERR_UNSUPPORTED;

  char *ws = static_cast<char *>(workspace);
  size_t ws_left = workspace_bytes;

  // sorted == 0: sort the edge ids by dst row (stable LSD radix sort keeps the edge order inside a
  // row), then run the same deterministic kernels with the permutation as an extra gather.  The
  // reference uses an all-atomic kernel here (index_scatter_kernel.cuh:204-263).
  const int64_t *d_dst = dst_index, *d_src = src_index;
  if (!sorted && weight) return GEOT_ERR_UNSUPPORTED;  // weights follow the edge order: sorted input only
  if (!sorted && reduce == GEOT_SUM && dtype == GEOT_F32 && !opts && g_unsorted_mode == 0 && env_int("GEOT_B200_UNSORTED_SORT", 0) == 0) {
    // fp32 sum: clear dst, then one pass of vector atomics (see scatter_add_kernel)
    CUDA_TRY(cudaMemsetAsync(dst, 0, (size_t)S * (size_t)W * sizeof(float), stream));
    const bool vec = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
    const int64_t pieces = vec ? W / 4 : W;
    if (pieces > 0x7fffffffLL) return GEOT_ERR_UNSUPPORTED;
    int shift = -1;
    if ((pieces & (pieces - 1)) == 0) { shift = 0; while ((1LL << shift) < pieces) ++shift; }
    const int64_t total = E * pieces;
    const int64_t need = (total + 256LL * kScatterUnroll - 1) / (256LL * kScatterUnroll);
    const unsigned blocks = (unsigned)std::min<int64_t>(need, 148LL * 8);
    if (vec)
      scatter_add_kernel<float4><<<blocks, 256, 0, stream>>>(static_cast<const float4 *>(src), src_index, dst_index,
                                                             static_cast<float *>(dst), E, (int)pieces, shift, S);
    else
      scatter_add_kernel<float><<<blocks, 256, 0, stream>>>(static_cast<const float *>(src), src_index, dst_index,
                                                            static_cast<float *>(dst), E, (int)pieces, shift, S);
    CUDA_TRY(cudaGetLastError());
    return GEOT_OK;
  }
  if (!sorted) {
    const size_t ebytes = align256((size_t)E * 8);
    size_t cub_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int64_t *)nullptr, (int64_t *)nullptr,
                                    (const int64_t *)nullptr, (int64_t *)nullptr, E);
    if (ws_left < 4 * ebytes + align256(cub_bytes)) return GEOT_ERR_WORKSPACE;
    int64_t *keys_out = reinterpret_cast<int64_t *>(ws);
    int64_t *iota = reinterpret_cast<int64_t *>(ws + ebytes);
    int64_t *perm = reinterpret_cast<int64_t *>(ws + 2 * ebytes);
    int64_t *src_perm = reinterpret_cast<int64_t *>(ws + 3 * ebytes);
    void *cub_tmp = ws + 4 * ebytes;
    ws += 4 * ebytes + align256(cub_bytes);
    ws_left -= 4 * ebytes + align256(cub_bytes);
    const unsigned nb = (unsigned)((E + 255) / 256);
    iota_kernel<<<nb, 256, 0, stream>>>(iota, E);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, dst_index, keys_out, iota, perm, E, 0, bits_for(S), stream));
    if (src_index) {
      gather_index_kernel<<<nb, 256, 0, stream>>>(perm, src_index, src_perm, E);
      CUDA_TRY(cudaGetLastError());
      d_src = src_perm;
    } else {
      d_src = perm;
    }
    d_dst = keys_out;
    plan = nullptr;
  }

  const bool aligned = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
  const Config cfg = choose_config(E, W, F, dtype, aligned, d_src != nullptr);
  Workspace w = carve(ws, cfg.n_tiles, W, dtype);
  if (w.bytes > ws_left) return GEOT_ERR_WORKSPACE;
  // The lean ring carries dst row ids and src row ids (index_scatter: edge ids) as 32-bit values.  A ring row is >= 128
  // bytes, so neither can reach 2^32 on a 180 GB device -- but the launcher does not rely on that: beyond 32 bits the
  // first-generation ring (64-bit offsets) is selected.
  const bool ids_fit_32 = S <= 0xffffffffLL && (d_src != nullptr || E <= 0xffffffffLL);

  // Rows that receive no edge must read 0.  The kernels store every non-empty row exactly once; the rows in between
  // are zeroed by zero_empty_rows_kernel when the call comes with a plan, else INSIDE the main kernel by the group that
  // sees the jump in the (sorted) index -- either way there is no memset of dst (the reference clears all of it first:
  // csrc/gather_scatter.cpp:27-30).  Only a tail of rows beyond the largest index that the plan knows about is cleared
  // with a memset in the plan-less form (normally empty: S = index[-1] + 1).
  int zero_gaps = 0;
  int64_t fill_lo = ex.fill_lo, fill_hi = ex.fill_hi < 0 ? S : ex.fill_hi;
  if (ex.clear_mode == 0 && !accumulate && !(plan && !plan->has_gaps && plan->S == S)) {
    zero_gaps = 1;
    // with a plan of the whole call the empty rows are known up front: one small kernel zeroes exactly those and the
    // main kernel stays the plain instantiation (GEOT_B200_ZERO_IN_KERNEL=1: fill inside the main kernel instead, A/B)
    if (plan && plan->is_sorted && plan->rowptr && plan->S <= S && ex.fill_hi < 0 && ex.fill_lo == 0 &&
        env_int("GEOT_B200_ZERO_IN_KERNEL", 0) == 0) {
      const size_t row_bytes = (size_t)W * dtype_size(dtype);
      const int vec16 = (row_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) ? 1 : 0;
      const unsigned nb = (unsigned)std::min<int64_t>((S + 255) / 256, 148 * 8);
      zero_empty_rows_kernel<<<nb, 256, 0, stream>>>(plan->rowptr, plan->S, S, (int64_t)row_bytes, static_cast<char *>(dst), vec16);
      CUDA_TRY(cudaGetLastError());
      zero_gaps = 0;
    }
  }
  if (zero_gaps) {
    if (plan && plan->is_sorted && plan->max_row + 1 < fill_hi) {
      const size_t row_bytes = (size_t)W * dtype_size(dtype);
      CUDA_TRY(cudaMemsetAsync(static_cast<char *>(dst) + (size_t)(plan->max_row + 1) * row_bytes, 0,
                               (size_t)(fill_hi - plan->max_row - 1) * row_bytes, stream));
      fill_hi = plan->max_row + 1;
    }
  }

  geot::Params p;
  p.src = src;
  p.src_index = d_src;
  p.dst_index = d_dst;
  p.weight = weight;
  p.dst = dst;
  p.E = E;
  p.W = W;
  p.F = F;
  p.ws_e = 1;
  p.ws_h = 0;
  if (weight_layout == GEOT_W_EDGE_HEAD) { p.ws_e = H; p.ws_h = 1; }
  if (weight_layout == GEOT_W_HEAD_EDGE) { p.ws_e = 1; p.ws_h = E; }
  geot::Shape shape = cfg.shape;
  if (!ids_fit_32 && (shape.pf & geot::kLeanFlag)) shape.pf = (shape.vpl == 1) ? 3 : 2;
  shape.wm = !weight ? geot::WM_NONE : (H == 1 ? geot::WM_EDGE : geot::WM_GENERIC);
  p.mean = (reduce == GEOT_MEAN);
  p.accumulate = accumulate ? 1 : 0;
  p.zero_gaps = zero_gaps;
  p.fill_lo = fill_lo;
  p.fill_hi = fill_hi;
  p.mean_rowptr = mean_rowptr;
  p.edge_perm = edge_perm;
  p.chunk_edges = cfg.chunk_edges;
  p.n_tiles = cfg.n_tiles;
  p.carry_head = w.carry_head;
  p.carry_tail = w.carry_tail;
  p.head_cnt = w.head_cnt;
  p.tail_cnt = w.tail_cnt;
  p.tail_row = w.tail_row;
  p.flags = w.flags;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (g_prof.n > 0) {
    const int slot = (int)(g_prof.calls % g_prof.n);
    ev0 = g_prof.start[slot];
    ev1 = g_prof.stop[slot];
    g_prof.calls += 1;
  }
  CUDA_TRY(launch(p, shape, stream, ev0, ev1));
  return GEOT_OK;
}

extern "C" {

int geot_b200_segment_reduce(const void *src, const int64_t *src_index, const int64_t *dst_index,
                             const void *weight, void *dst, int64_t E, int64_t S, int64_t H, int64_t F,
                             int dtype, int reduce, int weight_layout, int sorted, const geot_plan_t *plan,
                             void *workspace, size_t workspace_bytes, cudaStream_t stream) {
  return segment_reduce_impl(src, src_index, dst_index, weight, dst, E, S, H, F, dtype, reduce, weight_layout, sorted,
                             plan, workspace, workspace_bytes, stream, nullptr, Extra());
}

size_t geot_b200_src_blocks_workspace_bytes(const geot_src_blocks_t *blocks, int64_t W, int dtype) {
  if (!blocks) return 256;
  size_t best = 256;
  for (int b = 0; b < blocks->n_blocks; ++b)
    best = std::max(best, geot_b200_workspace_bytes(blocks->bounds[b + 1] - blocks->bounds[b], W, dtype, 1));
  return best;
}

int geot_b200_segment_reduce_ex(const void *src, const int64_t *src_index, const int64_t *dst_index,
                                const void *weight, void *dst, int64_t E, int64_t S, int64_t H, int64_t F,
                                int dtype, int reduce, int weight_layout, int sorted, const geot_plan_t *plan,
                                void *workspace, size_t workspace_bytes, cudaStream_t stream,
                                const geot_reduce_opts_t *opts) {
  if (opts && opts->struct_size != sizeof(geot_reduce_opts_t)) return GEOT_ERR_INVALID_ARG;
  if (!opts || !opts->src_blocks)
    return segment_reduce_impl(src, src_index, dst_index, weight, dst, E, S, H, F, dtype, reduce, weight_layout, sorted,
                               plan, workspace, workspace_bytes, stream, opts, Extra());
  // src-blocked: one pass per block of the regrouped list; pass 0 writes every row of dst (unless the caller already
  // accumulates), the others add their partial sums.  The caller's weights are read through the permutation.
  const geot_src_blocks_t *bl = opts->src_blocks;
  if (!src_index || bl->E != E || bl->n_blocks < 1 || bl->n_blocks > GEOT_MAX_SRC_BLOCKS || !sorted) return GEOT_ERR_INVALID_ARG;
  if ((reduce != GEOT_SUM && reduce != GEOT_MEAN) || opts->edge_perm) return GEOT_ERR_UNSUPPORTED;
  if (weight && weight_layout != GEOT_W_EDGE) return GEOT_ERR_UNSUPPORTED;
  const int64_t *mean_rowptr = opts->mean_rowptr;
  if (reduce == GEOT_MEAN && !mean_rowptr) {
    if (!plan || !plan->rowptr || plan->S != S) return GEOT_ERR_INVALID_ARG;     // the degrees of the complete list
    mean_rowptr = plan->rowptr;
  }
  bool first = true;
  for (int b = 0; b < bl->n_blocks; ++b) {
    const int64_t e0 = bl->bounds[b], n = bl->bounds[b + 1] - e0;
    if (n <= 0) continue;
    geot_reduce_opts_t o;
    memset(&o, 0, sizeof(o));
    o.struct_size = sizeof(o);
    o.accumulate = (opts->accumulate || !first) ? 1 : 0;
    o.edge_perm = weight ? bl->edge_perm + e0 : nullptr;
    o.mean_rowptr = mean_rowptr;
    const int rc = segment_reduce_impl(src, bl->src_index + e0, bl->dst_index + e0, weight, dst, n, S, H, F, dtype, reduce,
                                       weight_layout, 1, nullptr, workspace, workspace_bytes, stream, &o, Extra());
    if (rc != GEOT_OK) return rc;
    first = false;
  }
  return GEOT_OK;
}

int geot_b200_index_scatter(const void *src, const int64_t *index, void *dst, int64_t E, int64_t S, int64_t F,
                            int dtype, int reduce, int sorted, const geot_plan_t *plan, void *workspace,
                            size_t workspace_bytes, cudaStream_t stream) {
  return geot_b200_segment_reduce(src, nullptr, index, nullptr, dst, E, S, 1, F, dtype, reduce, GEOT_W_NONE, sorted,
                                  plan, workspace, workspace_bytes, stream);
}

int geot_b200_gather_scatter(const void *src, const int64_t *src_index, const int64_t *dst_index, void *dst,
                             int64_t E, int64_t S, int64_t F, int dtype, int reduce, const geot_plan_t *plan,
                             void *workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!src_index) return GEOT_ERR_INVALID_ARG;
  return geot_b200_segment_reduce(src, src_index, dst_index, nullptr, dst, E, S, 1, F, dtype, reduce, GEOT_W_NONE, 1,
                                  plan, workspace, workspace_bytes, stream);
}

int geot_b200_gather_weight_scatter(const void *src, const int64_t *src_index, const int64_t *dst_index,
                                    const void *weight, void *dst, int64_t E, int64_t S, int64_t F, int dtype,
                                    int reduce, const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                                    cudaStream_t stream) {
  if (!src_index || !weight) return GEOT_ERR_INVALID_ARG;
  return geot_b200_segment_reduce(src, src_index, dst_index, weight, dst, E, S, 1, F, dtype, reduce, GEOT_W_EDGE, 1,
                                  plan, workspace, workspace_bytes, stream);
}

int geot_b200_mh_spmm(const void *src, const int64_t *src_index, const int64_t *dst_index, const void *weight,
                      void *dst, int64_t E, int64_t S, int64_t H, int64_t F, int dtype, int reduce, int weight_layout,
                      const geot_plan_t *plan, void *workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!src_index || !weight) return GEOT_ERR_INVALID_ARG;
  if (weight_layout != GEOT_W_EDGE_HEAD && weight_layout != GEOT_W_HEAD_EDGE) return GEOT_ERR_INVALID_ARG;
  return geot_b200_segment_reduce(src, src_index, dst_index, weight, dst, E, S, H, F, dtype, reduce, weight_layout, 1,
                                  plan, workspace, workspace_bytes, stream);
}

int geot_b200_set_unsorted_mode(int mode) {
  if (mode != 0 && mode != 1) return GEOT_ERR_INVALID_ARG;
  g_unsorted_mode = mode;
  return GEOT_OK;
}

int geot_b200_profile_enable(int n) {
  if (n < 0) return GEOT_ERR_INVALID_ARG;
  for (int i = 0; i < g_prof.n; ++i) { cudaEventDestroy(g_prof.start[i]); cudaEventDestroy(g_prof.stop[i]); }
  delete[] g_prof.start; delete[] g_prof.stop;
  g_prof = Profile();
  if (n == 0) return GEOT_OK;
  g_prof.start = new cudaEvent_t[n];
  g_prof.stop = new cudaEvent_t[n];
  for (int i = 0; i < n; ++i) { CUDA_TRY(cudaEventCreate(&g_prof.start[i])); CUDA_TRY(cudaEventCreate(&g_prof.stop[i])); }
  g_prof.n = n;
  return GEOT_OK;
}

int geot_b200_profile_read(float *ms, int capacity, int *count) {
  if (!ms || !count) return GEOT_ERR_INVALID_ARG;
  const long long have = std::min<long long>(g_prof.calls, g_prof.n);
  const int k = (int)std::min<long long>(have, capacity);
  for (int i = 0; i < k; ++i) {
    const int slot = (int)((g_prof.calls - k + i) % g_prof.n);
    CUDA_TRY(cudaEventSynchronize(g_prof.stop[slot]));
    CUDA_TRY(cudaEventElapsedTime(&ms[i], g_prof.start[slot], g_prof.stop[slot]));
  }
  *count = k;
  return GEOT_OK;
}

}  // extern "C"
