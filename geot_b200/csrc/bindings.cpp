// bindings.cpp -- thin torch-extension bindings over the C ABI (include/geot_b200.h).
//
// Registers the reference's operator schemas under library `geot` (csrc/index_scatter.cpp:43-47,
// gather_scatter.cpp:16-17, gather_weight_scatter.cpp:12-14, mh_spmm.cpp:23), CUDA only: there is
// no CPU implementation and no fallback.  Everything here is tensor <-> pointer translation,
// output allocation and status -> TORCH_CHECK; the arithmetic lives behind the C ABI.
//
// Differences from the reference bindings, on purpose (SURVEY.md Appendix A):
//   * `index[-1].item()` per call (csrc/gather_scatter.cpp:27) is replaced by a cached
//     format_preprocess plan keyed on the index tensor's storage + version: the first call on a
//     graph synchronises once, later calls not at all;
//   * the output is allocated uninitialised (the kernels own every row) instead of torch::zeros;
//   * kernels run on the current stream under a device guard, not on the legacy default stream;
//   * `reduce` and `dim` are honoured (the reference validates and then ignores both).
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <cstdlib>
#include <cstring>
#include <limits>
#include <list>
#include <mutex>
#include <string>
#include <tuple>

#include "../../include/geot_b200.h"

namespace {

// ---- helpers ------------------------------------------------------------------------------------
// Same accepted strings and message as csrc/reduceutils.h:5-22.
int reduce_enum(c10::string_view reduce) {
  if (reduce == "max" || reduce == "amax") return GEOT_MAX;
  if (reduce == "mean") return GEOT_MEAN;
  if (reduce == "min" || reduce == "amin") return GEOT_MIN;
  if (reduce == "sum") return GEOT_SUM;
  if (reduce == "prod") return GEOT_PROD;
  TORCH_CHECK(false, "reduce argument must be either sum, prod, mean, amax or amin, got ", reduce);
}

int dtype_enum(const at::Tensor &t) {
  switch (t.scalar_type()) {
    case at::kFloat: return GEOT_F32;
    case at::kDouble: return GEOT_F64;
    case at::kBFloat16: return GEOT_BF16;
    case at::kHalf: return GEOT_F16;
    default: TORCH_CHECK(false, "geot: unsupported dtype ", t.scalar_type(), " (float32, float64, bfloat16, float16)");
  }
}

void check_status(int st, const char *what) {
  if (st == GEOT_OK) return;
  if (st == GEOT_ERR_CUDA) TORCH_CHECK(false, "geot::", what, ": ", geot_b200_last_cuda_error());
  if (st == GEOT_ERR_EMPTY) TORCH_CHECK(false, "geot::", what, ": index is empty (the output size is index[-1] + 1)");
  TORCH_CHECK(false, "geot::", what, ": ", geot_b200_status_string(st));
}

void check_index(const at::Tensor &idx, const char *name) {
  TORCH_CHECK(idx.is_cuda(), "geot: ", name, " must be a CUDA tensor (this build has no CPU path)");
  TORCH_CHECK(idx.scalar_type() == at::kLong, "geot: ", name, " must be int64");
}

// ---- plan cache -----------------------------------------------------------------------------------
// Keyed on (storage, offset, numel, version counter): a hit proves the bytes are the ones the plan
// was built from (the storage is still alive, so its address was not reused, and no in-place torch op
// touched it).  Small LRU; entries hold the plan's device buffer, not the index tensor.
struct PlanEntry {
  explicit PlanEntry(c10::weak_intrusive_ptr<c10::StorageImpl> s) : storage(std::move(s)) {}
  c10::weak_intrusive_ptr<c10::StorageImpl> storage;
  const void *storage_raw;
  int64_t offset, numel;
  uint32_t version;
  int device;
  at::Tensor buf;
  geot_plan_t plan;
};
std::mutex g_plan_mu;
std::list<PlanEntry> g_plans;
constexpr size_t kMaxPlans = 16;

uint32_t version_of(const at::Tensor &t) {
  return t.is_inference() ? 0u : t.unsafeGetTensorImpl()->version_counter().current_version();
}

// Returns a copy of the cached plan for dst_index (building it on a miss: one stream sync).
geot_plan_t get_plan(const at::Tensor &dst_index, at::Tensor *keepalive) {
  c10::StorageImpl *raw = dst_index.storage().unsafeGetStorageImpl();
  const int64_t off = dst_index.storage_offset(), n = dst_index.numel();
  const uint32_t ver = version_of(dst_index);
  const int dev = dst_index.get_device();
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto it = g_plans.begin(); it != g_plans.end();) {
      if (it->storage.expired()) {          // the index tensor is gone: its plan can never hit again
        it = g_plans.erase(it);
        continue;
      }
      if (it->storage_raw == raw && it->offset == off && it->numel == n && it->version == ver && it->device == dev) {
        g_plans.splice(g_plans.begin(), g_plans, it);
        *keepalive = it->buf;
        return it->plan;
      }
      ++it;
    }
  }
  auto stream = at::cuda::getCurrentCUDAStream();
  int64_t last = -1;
  check_status(geot_b200_index_last(dst_index.data_ptr<int64_t>(), n, &last, stream), "format_preprocess");
  TORCH_CHECK(last >= 0, "geot: negative index");
  const int64_t S = last + 1;
  const size_t bytes = geot_b200_plan_bytes(n, S);
  PlanEntry e(dst_index.storage().getWeakStorageImpl());
  e.buf = at::empty({(int64_t)bytes}, dst_index.options().dtype(at::kByte));
  check_status(geot_b200_format_preprocess(dst_index.data_ptr<int64_t>(), n, S, e.buf.data_ptr(), bytes, &e.plan, stream),
               "format_preprocess");
  e.storage_raw = raw;
  e.offset = off;
  e.numel = n;
  e.version = ver;
  e.device = dev;
  *keepalive = e.buf;
  geot_plan_t plan = e.plan;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    g_plans.push_front(std::move(e));
    while (g_plans.size() > kMaxPlans) g_plans.pop_back();
  }
  return plan;
}

// ---- src-block cache (geot_b200_src_blocks_build: the graph regrouped by src-row block for the L2) ----------------
// Keyed on both index tensors like the plan cache; an entry holds the regrouped list (20 bytes per edge).
struct BlocksEntry {
  c10::weak_intrusive_ptr<c10::StorageImpl> s_storage, d_storage;
  const void *s_raw, *d_raw;
  int64_t s_off, d_off, numel, n_src;
  uint32_t s_ver, d_ver;
  int device, n_blocks;
  at::Tensor buf;
  geot_src_blocks_t blocks;
  BlocksEntry(c10::weak_intrusive_ptr<c10::StorageImpl> a, c10::weak_intrusive_ptr<c10::StorageImpl> b)
      : s_storage(std::move(a)), d_storage(std::move(b)) {}
};
std::list<BlocksEntry> g_blocks;
constexpr size_t kMaxBlocks = 4;

geot_src_blocks_t get_src_blocks(const at::Tensor &src_index, const at::Tensor &dst_index, int64_t n_src, int n_blocks,
                                 at::Tensor *keepalive) {
  c10::StorageImpl *sr = src_index.storage().unsafeGetStorageImpl(), *dr = dst_index.storage().unsafeGetStorageImpl();
  const int64_t so = src_index.storage_offset(), d_o = dst_index.storage_offset(), n = dst_index.numel();
  const uint32_t sv = version_of(src_index), dv = version_of(dst_index);
  const int dev = dst_index.get_device();
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto it = g_blocks.begin(); it != g_blocks.end();) {
      if (it->s_storage.expired() || it->d_storage.expired()) {
        it = g_blocks.erase(it);
        continue;
      }
      if (it->s_raw == sr && it->d_raw == dr && it->s_off == so && it->d_off == d_o && it->numel == n && it->s_ver == sv &&
          it->d_ver == dv && it->device == dev && it->n_blocks == n_blocks && it->n_src == n_src) {
        g_blocks.splice(g_blocks.begin(), g_blocks, it);
        *keepalive = it->buf;
        return it->blocks;
      }
      ++it;
    }
  }
  auto stream = at::cuda::getCurrentCUDAStream();
  BlocksEntry e(src_index.storage().getWeakStorageImpl(), dst_index.storage().getWeakStorageImpl());
  const size_t bytes = geot_b200_src_blocks_bytes(n), sbytes = geot_b200_src_blocks_scratch_bytes(n);
  e.buf = at::empty({(int64_t)bytes}, dst_index.options().dtype(at::kByte));
  at::Tensor scratch = at::empty({(int64_t)sbytes}, dst_index.options().dtype(at::kByte));
  check_status(geot_b200_src_blocks_build(src_index.data_ptr<int64_t>(), dst_index.data_ptr<int64_t>(), n, n_src, n_blocks,
                                          e.buf.data_ptr(), bytes, scratch.data_ptr(), sbytes, &e.blocks, stream),
               "src_blocks_build");
  e.s_raw = sr; e.d_raw = dr; e.s_off = so; e.d_off = d_o; e.numel = n; e.n_src = n_src;
  e.s_ver = sv; e.d_ver = dv; e.device = dev; e.n_blocks = n_blocks;
  *keepalive = e.buf;
  geot_src_blocks_t blocks = e.blocks;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    g_blocks.push_front(std::move(e));
    while (g_blocks.size() > kMaxBlocks) g_blocks.pop_back();
  }
  return blocks;
}

void clear_csr_cache();
void clear_plan_cache() {
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    g_plans.clear();
    g_blocks.clear();
  }
  clear_csr_cache();
}

// ---- the one call every op funnels into ---------------------------------------------------------------
at::Tensor run(const char *what, const at::Tensor &src_in, const c10::optional<at::Tensor> &src_index_in,
               const at::Tensor &dst_index_in, const c10::optional<at::Tensor> &weight_in, int64_t H, int64_t F,
               int reduce, int weight_layout, bool sorted, std::vector<int64_t> out_shape, int64_t min_rows = 0) {
  c10::cuda::CUDAGuard guard(src_in.device());
  TORCH_CHECK(src_in.is_cuda(), "geot::", what, ": src must be a CUDA tensor (this build has no CPU path)");
  check_index(dst_index_in, "index");
  const at::Tensor src = src_in.contiguous();
  const at::Tensor dst_index = dst_index_in.contiguous();
  at::Tensor src_index, weight;
  if (src_index_in.has_value()) {
    check_index(*src_index_in, "src_index");
    src_index = src_index_in->contiguous();
    TORCH_CHECK(src_index.numel() == dst_index.numel(), "geot::", what, ": src_index and dst_index must have the same length");
  }
  if (weight_in.has_value()) {
    TORCH_CHECK(weight_in->scalar_type() == src.scalar_type(), "geot::", what, ": weight and src must have the same dtype");
    TORCH_CHECK(weight_in->device() == src.device(), "geot::", what, ": weight and src must be on the same device");
    weight = weight_in->contiguous();
  }
  TORCH_CHECK(dst_index.device() == src.device(), "geot::", what, ": index and src must be on the same device");
  const int64_t E = dst_index.numel();
  TORCH_CHECK(E > 0, "geot::", what, ": index is empty (the output size is index[-1] + 1)");
  // The fast path trusts src_index like the reference does (an id >= src.size(0) is an out-of-bounds read there too).
  // GEOT_B200_DEBUG=1 checks the range first: two reductions over the index and a host sync per call.
  if (src_index.defined()) {
    const char *dbg = std::getenv("GEOT_B200_DEBUG");
    if (dbg && dbg[0] == '1') {
      const int64_t lo = src_index.min().item<int64_t>(), hi = src_index.max().item<int64_t>();
      TORCH_CHECK(lo >= 0 && hi < src.size(0), "geot::", what, ": src_index out of range [0, ", src.size(0), "): min ", lo,
                  ", max ", hi);
      TORCH_CHECK(dst_index.min().item<int64_t>() >= 0, "geot::", what, ": negative dst index");
    }
  }
  const int dtype = dtype_enum(src);
  auto stream = at::cuda::getCurrentCUDAStream();

  geot_plan_t plan;
  const geot_plan_t *plan_ptr = nullptr;
  at::Tensor plan_buf;
  int64_t S;
  plan = get_plan(dst_index, &plan_buf);        // cached per index tensor: no pass over the index, no sync on later calls
  if (sorted) TORCH_CHECK(plan.is_sorted, "geot::", what, ": index is not sorted (pass sorted=False to index_scatter)");
  if (plan.is_sorted) {
    // sorted=False with an index that IS sorted -- what the reference's own test and benchmark pass
    // (test/test_index_scatter.py:9-14, benchmark/bench_index_scatter.py:32) -- takes the sorted kernels
    sorted = true;
    plan_ptr = &plan;
    S = plan.S;
  } else {
    S = plan.max_row + 1;                       // (the plan's row pointers mean nothing for an unsorted index: not passed on)
    check_status(geot_b200_set_unsorted_mode(at::globalContext().deterministicAlgorithms() ? 1 : 0), what);
  }
  // min_rows > S: the caller wants trailing rows that no edge reaches (csr_gws); they are zero-filled here and the
  // kernels see the [S, W] prefix
  out_shape[0] = std::max(S, min_rows);
  at::Tensor out = at::empty(out_shape, src.options());
  if (min_rows > S) out.narrow(0, S, min_rows - S).zero_();
  const int64_t W = H * F;
  size_t ws_bytes = geot_b200_workspace_bytes(E, W, dtype, sorted ? 1 : 0);
  // src-row blocking for the L2 (high-reuse graphs whose src matrix exceeds what the L2 keeps): the graph regrouped
  // once, cached next to the plan.  GEOT_B200_SRC_BLOCKS: unset / 0 = the library's suggestion, 1 = off, n = n blocks.
  geot_src_blocks_t blocks;
  at::Tensor blocks_buf;
  geot_reduce_opts_t opts;
  memset(&opts, 0, sizeof(opts));
  opts.struct_size = sizeof(opts);
  const bool blockable = sorted && src_index.defined() && (reduce == GEOT_SUM || reduce == GEOT_MEAN) &&
                         (weight_layout == GEOT_W_NONE || weight_layout == GEOT_W_EDGE);
  if (blockable) {
    const char *env = std::getenv("GEOT_B200_SRC_BLOCKS");
    int nb = (env && env[0]) ? std::atoi(env) : 0;
    // (automatic only for 4- / 8-byte elements: a 16-bit output would be rounded once per pass)
    if (nb <= 0) nb = src.element_size() >= 4 ? geot_b200_src_blocks_suggest(E, S, src.size(0), W * (int64_t)src.element_size()) : 1;
    if (nb > 1 && nb <= GEOT_MAX_SRC_BLOCKS) {
      blocks = get_src_blocks(src_index, dst_index, src.size(0), nb, &blocks_buf);
      opts.src_blocks = &blocks;
      ws_bytes = std::max(ws_bytes, geot_b200_src_blocks_workspace_bytes(&blocks, W, dtype));
    }
  }
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, src.options().dtype(at::kByte));
  const int st = geot_b200_segment_reduce_ex(
      src.data_ptr(), src_index.defined() ? src_index.data_ptr<int64_t>() : nullptr, dst_index.data_ptr<int64_t>(),
      weight.defined() ? weight.data_ptr() : nullptr, out.data_ptr(), E, S, H, F, dtype, reduce, weight_layout,
      sorted ? 1 : 0, plan_ptr, ws.data_ptr(), ws_bytes, stream, opts.src_blocks ? &opts : nullptr);
  check_status(st, what);
  return out;
}

// ---- ops ---------------------------------------------------------------------------------------------
// geot::index_scatter -- csrc/index_scatter.cpp:26-39 + csrc/cuda/index_scatter_cuda.cu:86-105
at::Tensor index_scatter_cuda_impl(int64_t dim, at::Tensor index, at::Tensor src, c10::string_view reduce, bool sorted) {
  TORCH_CHECK(dim >= 0 && dim < src.dim(), "dim must be non-negative and less than input dimensions");
  TORCH_CHECK(index.dim() == 1, "index must be 1 dimensional");
  TORCH_CHECK(src.size(dim) == index.size(0), "index length must be equal to src dimension size");
  const int red = reduce_enum(reduce);
  TORCH_CHECK(index.size(0) > 0, "geot::index_scatter: index is empty (the output size is index[-1] + 1)");
  at::Tensor s = (dim == 0) ? src : src.movedim(dim, 0);
  s = s.contiguous();
  const int64_t E = index.size(0);
  const int64_t F = E > 0 ? s.numel() / E : 0;
  TORCH_CHECK(F > 0, "geot::index_scatter: src has no elements");
  at::Tensor out = run("index_scatter", s, c10::nullopt, index, c10::nullopt, 1, F, red, GEOT_W_NONE, sorted, s.sizes().vec());
  return (dim == 0) ? out : out.movedim(0, dim);
}

at::Tensor gather_scatter_reduce(at::Tensor src_index, at::Tensor dst_index, at::Tensor src, c10::string_view reduce) {
  // checks and messages: csrc/cuda/gather_scatter_cuda.cu:18-22
  TORCH_CHECK(src_index.dim() == dst_index.dim() && src_index.dim() == 1, "src_index and dst_index must be 1 dimensional");
  TORCH_CHECK(src.dim() == 2, "src must be 2 dimensional");
  return run("gather_scatter", src, src_index, dst_index, c10::nullopt, 1, src.size(1), reduce_enum(reduce), GEOT_W_NONE, true,
             src.sizes().vec());
}
// geot::gather_scatter_impl -- csrc/gather_scatter.cpp:25-34 (sum)
at::Tensor gather_scatter_impl(at::Tensor src_index, at::Tensor dst_index, at::Tensor src) {
  return gather_scatter_reduce(src_index, dst_index, src, "sum");
}

at::Tensor gather_weight_scatter_reduce(at::Tensor src_index, at::Tensor dst_index, at::Tensor weight, at::Tensor src,
                                        c10::string_view reduce) {
  // checks: csrc/cuda/gather_weight_scatter_cuda.cu:27-33
  TORCH_CHECK(src_index.dim() == dst_index.dim() && src_index.dim() == 1, "src_index and dst_index must be 1 dimensional");
  TORCH_CHECK(src.dim() == 2, "src must be 2 dimensional");
  TORCH_CHECK(weight.dim() == 1 && weight.size(0) == dst_index.size(0), "weight must be 1 dimensional with one entry per edge");
  return run("gather_weight_scatter", src, src_index, dst_index, weight, 1, src.size(1), reduce_enum(reduce), GEOT_W_EDGE, true,
             src.sizes().vec());
}
// geot::gather_weight_scatter_impl -- csrc/gather_weight_scatter.cpp:22-34 (hard-codes "sum", :31)
at::Tensor gather_weight_scatter_impl(at::Tensor src_index, at::Tensor dst_index, at::Tensor weight, at::Tensor src) {
  return gather_weight_scatter_reduce(src_index, dst_index, weight, src, "sum");
}

// geot::mh_spmm -- csrc/mh_spmm.cpp:10-23 + csrc/cuda/mh_spmm_cuda.cu:20-38
at::Tensor mh_spmm_impl(at::Tensor src_index, at::Tensor dst_index, at::Tensor weight, at::Tensor src, c10::string_view reduce) {
  TORCH_CHECK(src_index.dim() == dst_index.dim() && src_index.dim() == 1, "src_index and dst_index must be 1 dimensional");
  TORCH_CHECK(src.dim() == 3, "src must be 3 dimensional");
  const int red = reduce_enum(reduce);
  const int64_t E = src_index.size(0), H = src.size(1), F = src.size(2);
  // weight layout by shape, [E,H] first -- wrapper/mh_spmm_base.h:38-49
  int layout;
  if (weight.dim() == 2 && weight.size(0) == E && weight.size(1) == H) layout = GEOT_W_EDGE_HEAD;
  else if (weight.dim() == 2 && weight.size(1) == E && weight.size(0) == H) layout = GEOT_W_HEAD_EDGE;
  else throw std::runtime_error("Invalid weight size");
  return run("mh_spmm", src, src_index, dst_index, weight, H, F, red, layout, true, src.sizes().vec());
}

// geot::format_preprocess -> (rowptr [S+1] int64 on device, stats [6] int64 on CPU:
// E, S, num_segments, max_degree, is_sorted, has_gaps)
std::tuple<at::Tensor, at::Tensor> format_preprocess(at::Tensor dst_index) {
  check_index(dst_index, "dst_index");
  TORCH_CHECK(dst_index.dim() == 1, "index must be 1 dimensional");
  TORCH_CHECK(dst_index.numel() > 0, "geot::format_preprocess: index is empty");
  c10::cuda::CUDAGuard guard(dst_index.device());
  at::Tensor idx = dst_index.contiguous();
  at::Tensor buf;
  geot_plan_t plan = get_plan(idx, &buf);
  at::Tensor rowptr = at::from_blob(const_cast<int64_t *>(plan.rowptr), {plan.S + 1},
                                    [buf](void *) mutable { buf.reset(); }, idx.options());
  at::Tensor stats = at::empty({6}, at::TensorOptions().dtype(at::kLong));
  int64_t *s = stats.data_ptr<int64_t>();
  s[0] = plan.E; s[1] = plan.S; s[2] = plan.num_segments; s[3] = plan.max_degree; s[4] = plan.is_sorted; s[5] = plan.has_gaps;
  return std::make_tuple(rowptr, stats);
}

// geot::plan_shards -> CPU int64 [2, parts+1]: row bounds, edge bounds
at::Tensor plan_shards(at::Tensor dst_index, int64_t parts) {
  check_index(dst_index, "dst_index");
  c10::cuda::CUDAGuard guard(dst_index.device());
  at::Tensor idx = dst_index.contiguous();
  at::Tensor buf;
  geot_plan_t plan = get_plan(idx, &buf);
  TORCH_CHECK(plan.is_sorted, "geot::plan_shards: index is not sorted");
  at::Tensor out = at::empty({2, parts + 1}, at::TensorOptions().dtype(at::kLong));
  check_status(geot_b200_plan_shards(&plan, (int)parts, out.data_ptr<int64_t>(), out.data_ptr<int64_t>() + (parts + 1),
                                     at::cuda::getCurrentCUDAStream()),
               "plan_shards");
  return out;
}

// geot::sddmm_coo_impl -- csrc/gather_weight_scatter.cpp:36-44 + csrc/cuda/gather_weight_scatter_cuda.cu:41-62:
// out[e] = <mat_1[dst_index[e]], mat_2[src_index[e]]> (row = dst_index, col = src_index).  The reference
// narrows the indices to int32 and is fp32 only; here int64 / int32 indices and all four dtypes.
at::Tensor sddmm_coo_impl(at::Tensor src_index, at::Tensor dst_index, at::Tensor mat_1, at::Tensor mat_2) {
  TORCH_CHECK(mat_1.is_cuda() && mat_2.is_cuda(), "geot::sddmm_coo: mat_1 and mat_2 must be CUDA tensors (this build has no CPU path)");
  TORCH_CHECK(src_index.dim() == 1 && dst_index.dim() == 1 && src_index.numel() == dst_index.numel(),
              "src_index and dst_index must be 1 dimensional and of the same length");
  TORCH_CHECK(mat_1.dim() == 2 && mat_2.dim() == 2 && mat_1.size(1) == mat_2.size(1), "mat_1 and mat_2 must be 2 dimensional with the same width");
  TORCH_CHECK(mat_1.scalar_type() == mat_2.scalar_type(), "mat_1 and mat_2 must have the same dtype");
  c10::cuda::CUDAGuard guard(mat_1.device());
  const at::Tensor col = src_index.to(at::kLong).contiguous(), row = dst_index.to(at::kLong).contiguous();
  TORCH_CHECK(row.is_cuda() && col.is_cuda(), "geot::sddmm_coo: indices must be CUDA tensors");
  const at::Tensor a = mat_1.contiguous(), b = mat_2.contiguous();
  at::Tensor out = at::empty({row.numel()}, a.options());
  check_status(geot_b200_sddmm_coo(a.data_ptr(), row.data_ptr<int64_t>(), b.data_ptr(), col.data_ptr<int64_t>(), out.data_ptr(),
                                   row.numel(), a.size(1), dtype_enum(a), at::cuda::getCurrentCUDAStream()),
               "sddmm_coo");
  return out;
}

// geot::sddmm_mh_impl -- the weight gradient of mh_spmm: out[e, h] = <mat_1[dst_index[e], h, :], mat_2[src_index[e], h, :]>,
// [E, H], or [H, E] with head_major (the two weight layouts of mh_spmm).  Checks as sddmm_coo_impl.
at::Tensor sddmm_mh_impl(at::Tensor src_index, at::Tensor dst_index, at::Tensor mat_1, at::Tensor mat_2, bool head_major) {
  TORCH_CHECK(mat_1.is_cuda() && mat_2.is_cuda(), "geot::sddmm_mh: mat_1 and mat_2 must be CUDA tensors (this build has no CPU path)");
  TORCH_CHECK(src_index.dim() == 1 && dst_index.dim() == 1 && src_index.numel() == dst_index.numel(),
              "src_index and dst_index must be 1 dimensional and of the same length");
  TORCH_CHECK(mat_1.dim() == 3 && mat_2.dim() == 3 && mat_1.size(1) == mat_2.size(1) && mat_1.size(2) == mat_2.size(2),
              "mat_1 and mat_2 must be 3 dimensional [N, H, F] with the same H and F");
  TORCH_CHECK(mat_1.scalar_type() == mat_2.scalar_type(), "mat_1 and mat_2 must have the same dtype");
  c10::cuda::CUDAGuard guard(mat_1.device());
  const at::Tensor col = src_index.to(at::kLong).contiguous(), row = dst_index.to(at::kLong).contiguous();
  TORCH_CHECK(row.is_cuda() && col.is_cuda(), "geot::sddmm_mh: indices must be CUDA tensors");
  const at::Tensor a = mat_1.contiguous(), b = mat_2.contiguous();
  const int64_t E = row.numel(), H = a.size(1), F = a.size(2);
  TORCH_CHECK(H > 0 && F > 0, "geot::sddmm_mh: mat_1 and mat_2 must have at least one head and one feature");
  at::Tensor out = head_major ? at::empty({H, E}, a.options()) : at::empty({E, H}, a.options());
  check_status(geot_b200_sddmm_mh(a.data_ptr(), row.data_ptr<int64_t>(), b.data_ptr(), col.data_ptr<int64_t>(), out.data_ptr(), E,
                                  H, F, dtype_enum(a), head_major ? GEOT_W_HEAD_EDGE : GEOT_W_EDGE_HEAD,
                                  at::cuda::getCurrentCUDAStream()),
               "sddmm_mh");
  return out;
}

// ---- segment softmax -------------------------------------------------------------------------------------
// geot::segment_softmax / geot::segment_softmax_backward: src / out / grad [E] or [E, H] over a sorted int64 index [E].
// The plan comes from the cache (no sync after the first call on a graph); an index it reports unsorted is refused.
void check_softmax_operand(const at::Tensor &t, const at::Tensor &index, const char *what, const char *name) {
  TORCH_CHECK(t.is_cuda(), "geot::", what, ": ", name, " must be a CUDA tensor (this build has no CPU path)");
  TORCH_CHECK(t.dim() == 1 || t.dim() == 2, "geot::", what, ": ", name, " must be [E] or [E, H]");
  TORCH_CHECK(t.size(0) == index.size(0), "geot::", what, ": ", name, " must have one row per index entry");
  TORCH_CHECK(t.device() == index.device(), "geot::", what, ": ", name, " and index must be on the same device");
}

geot_plan_t softmax_plan(const at::Tensor &index, const char *what, at::Tensor *keepalive) {
  geot_plan_t plan = get_plan(index, keepalive);
  TORCH_CHECK(plan.is_sorted, "geot::", what, ": index must be sorted (non-decreasing)");
  return plan;
}

at::Tensor segment_softmax_impl(at::Tensor src, at::Tensor index) {
  check_index(index, "index");
  TORCH_CHECK(index.dim() == 1, "geot::segment_softmax: index must be 1 dimensional");
  check_softmax_operand(src, index, "segment_softmax", "src");
  const int dtype = dtype_enum(src);
  c10::cuda::CUDAGuard guard(src.device());
  const at::Tensor x = src.contiguous(), idx = index.contiguous();
  at::Tensor out = at::empty_like(x);
  const int64_t E = idx.numel(), H = E > 0 ? x.numel() / E : 0;
  if (E == 0 || H == 0) return out;
  at::Tensor plan_buf;
  const geot_plan_t plan = softmax_plan(idx, "segment_softmax", &plan_buf);
  const size_t ws_bytes = geot_b200_segment_softmax_workspace_bytes(E, H, dtype);
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, x.options().dtype(at::kByte));
  check_status(geot_b200_segment_softmax(x.data_ptr(), idx.data_ptr<int64_t>(), out.data_ptr(), E, H, dtype, &plan,
                                         ws.data_ptr(), ws_bytes, at::cuda::getCurrentCUDAStream()),
               "segment_softmax");
  return out;
}

at::Tensor segment_softmax_backward_impl(at::Tensor out, at::Tensor grad_out, at::Tensor index) {
  check_index(index, "index");
  TORCH_CHECK(index.dim() == 1, "geot::segment_softmax_backward: index must be 1 dimensional");
  check_softmax_operand(out, index, "segment_softmax_backward", "out");
  check_softmax_operand(grad_out, index, "segment_softmax_backward", "grad_out");
  TORCH_CHECK(out.sizes() == grad_out.sizes(), "geot::segment_softmax_backward: out and grad_out must have the same shape");
  TORCH_CHECK(out.scalar_type() == grad_out.scalar_type(), "geot::segment_softmax_backward: out and grad_out must have the same dtype");
  const int dtype = dtype_enum(out);
  c10::cuda::CUDAGuard guard(out.device());
  const at::Tensor y = out.contiguous(), g = grad_out.contiguous(), idx = index.contiguous();
  at::Tensor grad_src = at::empty_like(y);
  const int64_t E = idx.numel(), H = E > 0 ? y.numel() / E : 0;
  if (E == 0 || H == 0) return grad_src;
  at::Tensor plan_buf;
  const geot_plan_t plan = softmax_plan(idx, "segment_softmax_backward", &plan_buf);
  const size_t ws_bytes = geot_b200_segment_softmax_workspace_bytes(E, H, dtype);
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, y.options().dtype(at::kByte));
  check_status(geot_b200_segment_softmax_backward(y.data_ptr(), g.data_ptr(), idx.data_ptr<int64_t>(), grad_src.data_ptr(),
                                                  E, H, dtype, &plan, ws.data_ptr(), ws_bytes,
                                                  at::cuda::getCurrentCUDAStream()),
               "segment_softmax_backward");
  return grad_src;
}

// ---- GATv2 attention score ---------------------------------------------------------------------------------
// geot::gatv2_score: score[e, h] = sum_f att[h, f] * leaky_relu(x_l[src[e], h, f] + x_r[dst[e], h, f]), x_l [N_l, H, F],
// x_r [N_r, H, F], att [H, F], dst_index sorted (the plan cache says so; an unsorted index is refused).
void check_gatv2_operands(const at::Tensor &x_l, const at::Tensor &x_r, const at::Tensor &att, const at::Tensor &src_index,
                          const at::Tensor &dst_index, const char *what) {
  TORCH_CHECK(x_l.is_cuda() && x_r.is_cuda() && att.is_cuda(), "geot::", what,
              ": x_l, x_r and att must be CUDA tensors (this build has no CPU path)");
  check_index(src_index, "src_index");
  check_index(dst_index, "dst_index");
  TORCH_CHECK(src_index.dim() == 1 && dst_index.dim() == 1 && src_index.numel() == dst_index.numel(), "geot::", what,
              ": src_index and dst_index must be 1 dimensional and of the same length");
  TORCH_CHECK(x_l.dim() == 3 && x_r.dim() == 3 && x_l.size(1) == x_r.size(1) && x_l.size(2) == x_r.size(2), "geot::", what,
              ": x_l and x_r must be [N, H, F] with the same H and F");
  TORCH_CHECK(att.dim() == 2 && att.size(0) == x_l.size(1) && att.size(1) == x_l.size(2), "geot::", what, ": att must be [H, F]");
  TORCH_CHECK(x_l.size(1) > 0 && x_l.size(2) > 0, "geot::", what, ": x_l and x_r must have at least one head and one feature");
  TORCH_CHECK(x_l.scalar_type() == x_r.scalar_type() && att.scalar_type() == x_l.scalar_type(), "geot::", what,
              ": x_l, x_r and att must have the same dtype");
  const auto dev = x_l.device();
  TORCH_CHECK(x_r.device() == dev && att.device() == dev && src_index.device() == dev && dst_index.device() == dev, "geot::",
              what, ": all operands must be on the same device");
}

at::Tensor gatv2_score_impl(at::Tensor x_l, at::Tensor x_r, at::Tensor att, at::Tensor src_index, at::Tensor dst_index,
                            double negative_slope) {
  check_gatv2_operands(x_l, x_r, att, src_index, dst_index, "gatv2_score");
  const int dtype = dtype_enum(x_l);
  c10::cuda::CUDAGuard guard(x_l.device());
  const at::Tensor xl = x_l.contiguous(), xr = x_r.contiguous(), a = att.contiguous();
  const at::Tensor si = src_index.contiguous(), di = dst_index.contiguous();
  const int64_t E = di.numel(), H = xl.size(1), F = xl.size(2);
  at::Tensor out = at::empty({E, H}, xl.options());
  if (E == 0) return out;
  at::Tensor plan_buf;
  softmax_plan(di, "gatv2_score", &plan_buf);        // cached: refuses an unsorted dst_index
  check_status(geot_b200_gatv2_score(xl.data_ptr(), xr.data_ptr(), a.data_ptr(), si.data_ptr<int64_t>(), di.data_ptr<int64_t>(),
                                     out.data_ptr(), E, H, F, dtype, &negative_slope, at::cuda::getCurrentCUDAStream()),
               "gatv2_score");
  return out;
}

// geot::gatv2_score_backward -> (grad_x_l, grad_x_r, grad_att); a gradient not asked for comes back as an empty tensor.
// The dst pass (grad_x_r, grad_att) runs on the dst-sorted list; the src pass (grad_x_l) on the transposed list
// t_perm / t_dst_index (= src_index[t_perm], sorted) / t_src_index (= dst_index[t_perm]) with the grads carried into that
// order.  Both plans come from the plan cache.
void gatv2_pass(const at::Tensor &x_row, const at::Tensor &x_gat, const at::Tensor &att, const at::Tensor &g,
                const at::Tensor &row_index, const at::Tensor &gat_index, at::Tensor &grad_row, at::Tensor *grad_att,
                double slope) {
  at::Tensor plan_buf;
  const geot_plan_t plan = softmax_plan(row_index, "gatv2_score_backward", &plan_buf);
  const int64_t E = row_index.numel(), H = x_row.size(1), F = x_row.size(2);
  const int dtype = dtype_enum(x_row);
  const size_t ws_bytes = geot_b200_gatv2_grad_workspace_bytes(E, H, F, dtype);
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, x_row.options().dtype(at::kByte));
  check_status(geot_b200_gatv2_grad(x_row.data_ptr(), x_gat.data_ptr(), att.data_ptr(), g.data_ptr(), row_index.data_ptr<int64_t>(),
                                    gat_index.data_ptr<int64_t>(), &plan, grad_row.size(0), grad_row.data_ptr(),
                                    grad_att ? grad_att->data_ptr() : nullptr, E, H, F, dtype, &slope, ws.data_ptr(), ws_bytes,
                                    at::cuda::getCurrentCUDAStream()),
               "gatv2_score_backward");
}

std::tuple<at::Tensor, at::Tensor, at::Tensor> gatv2_score_backward_impl(
    at::Tensor grad, at::Tensor x_l, at::Tensor x_r, at::Tensor att, at::Tensor src_index, at::Tensor dst_index,
    at::Tensor t_perm, at::Tensor t_dst_index, at::Tensor t_src_index, double negative_slope, bool need_x_l, bool need_x_r,
    bool need_att) {
  check_gatv2_operands(x_l, x_r, att, src_index, dst_index, "gatv2_score_backward");
  const int64_t E = dst_index.numel(), H = x_l.size(1);
  TORCH_CHECK(grad.dim() == 2 && grad.size(0) == E && grad.size(1) == H, "geot::gatv2_score_backward: grad must be [E, H]");
  TORCH_CHECK(grad.scalar_type() == x_l.scalar_type() && grad.device() == x_l.device(),
              "geot::gatv2_score_backward: grad must have the dtype and device of x_l");
  c10::cuda::CUDAGuard guard(x_l.device());
  const at::Tensor xl = x_l.contiguous(), xr = x_r.contiguous(), a = att.contiguous(), g = grad.contiguous();
  at::Tensor gl = need_x_l ? at::empty_like(xl) : at::empty({0}, xl.options());
  at::Tensor gr = need_x_r ? at::empty_like(xr) : at::empty({0}, xl.options());
  at::Tensor ga = need_att ? at::empty_like(a) : at::empty({0}, xl.options());
  if (E == 0) {            // no edge: every gradient is zero
    gl.zero_(); gr.zero_(); ga.zero_();
    return std::make_tuple(gl, gr, ga);
  }
  const at::Tensor si = src_index.contiguous(), di = dst_index.contiguous();
  if (need_x_r || need_att) {
    at::Tensor gr_buf = need_x_r ? gr : at::empty_like(xr);
    gatv2_pass(xr, xl, a, g, di, si, gr_buf, need_att ? &ga : nullptr, negative_slope);
  }
  if (need_x_l) {
    check_index(t_perm, "t_perm");
    check_index(t_dst_index, "t_dst_index");
    check_index(t_src_index, "t_src_index");
    TORCH_CHECK(t_perm.numel() == E && t_dst_index.numel() == E && t_src_index.numel() == E,
                "geot::gatv2_score_backward: the transposed edge list must have E entries");
    const at::Tensor perm = t_perm.contiguous(), tdi = t_dst_index.contiguous(), tsi = t_src_index.contiguous();
    at::Tensor gt = at::empty_like(g);
    check_status(geot_b200_permute_edges(g.data_ptr(), perm.data_ptr<int64_t>(), gt.data_ptr(), E, H * (int64_t)g.element_size(),
                                         at::cuda::getCurrentCUDAStream()),
                 "gatv2_score_backward");
    gatv2_pass(xl, xr, a, gt, tdi, tsi, gl, nullptr, negative_slope);
  }
  return std::make_tuple(gl, gr, ga);
}

// ---- dot-product graph attention ------------------------------------------------------------------------------------
// geot::graph_attention -> (out [N_dst, H, F], lse [N_dst, H] fp32 / fp64): q [N_dst, H, F] by dst, k / v [N_src, H, F]
// by src, dst_index sorted (the plan cache says so; an unsorted index is refused), N_dst = q.size(0).
void check_attention_operands(const at::Tensor &q, const at::Tensor &k, const at::Tensor &v, const at::Tensor &src_index,
                              const at::Tensor &dst_index, const char *what) {
  TORCH_CHECK(q.is_cuda() && k.is_cuda() && v.is_cuda(), "geot::", what,
              ": q, k and v must be CUDA tensors (this build has no CPU path)");
  check_index(src_index, "src_index");
  check_index(dst_index, "dst_index");
  TORCH_CHECK(src_index.dim() == 1 && dst_index.dim() == 1 && src_index.numel() == dst_index.numel(), "geot::", what,
              ": src_index and dst_index must be 1 dimensional and of the same length");
  TORCH_CHECK(q.dim() == 3 && k.dim() == 3 && v.dim() == 3 && k.sizes() == v.sizes() && q.size(1) == k.size(1) &&
                  q.size(2) == k.size(2),
              "geot::", what, ": q must be [N_dst, H, F] and k, v [N_src, H, F] with the same H and F");
  TORCH_CHECK(q.size(1) > 0 && q.size(2) > 0, "geot::", what, ": q, k and v must have at least one head and one feature");
  TORCH_CHECK(k.scalar_type() == q.scalar_type() && v.scalar_type() == q.scalar_type(), "geot::", what,
              ": q, k and v must have the same dtype");
  const auto dev = q.device();
  TORCH_CHECK(k.device() == dev && v.device() == dev && src_index.device() == dev && dst_index.device() == dev, "geot::",
              what, ": all operands must be on the same device");
}

at::ScalarType lse_type(const at::Tensor &q) { return q.scalar_type() == at::kDouble ? at::kDouble : at::kFloat; }

std::tuple<at::Tensor, at::Tensor> graph_attention_impl(at::Tensor q, at::Tensor k, at::Tensor v, at::Tensor src_index,
                                                        at::Tensor dst_index, double scale) {
  check_attention_operands(q, k, v, src_index, dst_index, "graph_attention");
  const int dtype = dtype_enum(q);
  c10::cuda::CUDAGuard guard(q.device());
  const at::Tensor qc = q.contiguous(), kc = k.contiguous(), vc = v.contiguous();
  const at::Tensor si = src_index.contiguous(), di = dst_index.contiguous();
  const int64_t E = di.numel(), N = qc.size(0), H = qc.size(1), F = qc.size(2);
  at::Tensor out = at::empty_like(qc);
  at::Tensor lse = at::empty({N, H}, qc.options().dtype(lse_type(qc)));
  if (E == 0) {            // no edge: every row is empty
    out.zero_();
    lse.fill_(-std::numeric_limits<double>::infinity());
    return std::make_tuple(out, lse);
  }
  at::Tensor plan_buf;
  const geot_plan_t plan = softmax_plan(di, "graph_attention", &plan_buf);
  TORCH_CHECK(plan.max_row < N, "geot::graph_attention: dst_index holds ", plan.max_row, " but q has ", N, " rows");
  const size_t ws_bytes = geot_b200_graph_attention_workspace_bytes(E, H, F, dtype);
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, qc.options().dtype(at::kByte));
  check_status(geot_b200_graph_attention(qc.data_ptr(), kc.data_ptr(), vc.data_ptr(), si.data_ptr<int64_t>(),
                                         di.data_ptr<int64_t>(), &plan, N, out.data_ptr(), lse.data_ptr(), E, H, F, dtype,
                                         &scale, ws.data_ptr(), ws_bytes, at::cuda::getCurrentCUDAStream()),
               "graph_attention");
  return std::make_tuple(out, lse);
}

// geot::graph_attention_backward -> (grad_q [N_dst, H, F], p [E, H], ds [E, H]): the dst pass of the backward; ds is
// scale * d loss / d score.  grad_k and grad_v are mh_spmm passes on the transposed edge list (attention.py).
std::tuple<at::Tensor, at::Tensor, at::Tensor> graph_attention_backward_impl(
    at::Tensor grad, at::Tensor q, at::Tensor k, at::Tensor v, at::Tensor out, at::Tensor lse, at::Tensor src_index,
    at::Tensor dst_index, double scale) {
  check_attention_operands(q, k, v, src_index, dst_index, "graph_attention_backward");
  TORCH_CHECK(grad.sizes() == q.sizes() && out.sizes() == q.sizes(),
              "geot::graph_attention_backward: grad and out must have the shape of q");
  TORCH_CHECK(grad.scalar_type() == q.scalar_type() && out.scalar_type() == q.scalar_type() && grad.device() == q.device() &&
                  out.device() == q.device(),
              "geot::graph_attention_backward: grad and out must have the dtype and device of q");
  TORCH_CHECK(lse.dim() == 2 && lse.size(0) == q.size(0) && lse.size(1) == q.size(1) && lse.scalar_type() == lse_type(q) &&
                  lse.device() == q.device(),
              "geot::graph_attention_backward: lse must be [N_dst, H] in the accumulator type");
  const int dtype = dtype_enum(q);
  c10::cuda::CUDAGuard guard(q.device());
  const at::Tensor qc = q.contiguous(), kc = k.contiguous(), vc = v.contiguous(), oc = out.contiguous(),
                   lc = lse.contiguous(), g = grad.contiguous();
  const at::Tensor si = src_index.contiguous(), di = dst_index.contiguous();
  const int64_t E = di.numel(), N = qc.size(0), H = qc.size(1), F = qc.size(2);
  at::Tensor grad_q = at::empty_like(qc);
  at::Tensor p = at::empty({E, H}, qc.options()), ds = at::empty({E, H}, qc.options());
  if (E == 0) {
    grad_q.zero_();
    return std::make_tuple(grad_q, p, ds);
  }
  at::Tensor plan_buf;
  const geot_plan_t plan = softmax_plan(di, "graph_attention_backward", &plan_buf);
  const size_t ws_bytes = geot_b200_graph_attention_grad_workspace_bytes(E, H, F, dtype);
  at::Tensor ws = at::empty({(int64_t)ws_bytes}, qc.options().dtype(at::kByte));
  check_status(geot_b200_graph_attention_grad(qc.data_ptr(), kc.data_ptr(), vc.data_ptr(), oc.data_ptr(), lc.data_ptr(),
                                              g.data_ptr(), si.data_ptr<int64_t>(), di.data_ptr<int64_t>(), &plan, N,
                                              grad_q.data_ptr(), p.data_ptr(), ds.data_ptr(), E, H, F, dtype, &scale,
                                              ws.data_ptr(), ws_bytes, at::cuda::getCurrentCUDAStream()),
               "graph_attention_backward");
  return std::make_tuple(grad_q, p, ds);
}

// ---- CSR entry point ------------------------------------------------------------------------------------
// Cache of the COO row index expanded from a CSR row pointer, keyed like the plans (storage + version).
struct CsrEntry {
  explicit CsrEntry(c10::weak_intrusive_ptr<c10::StorageImpl> s) : storage(std::move(s)) {}
  c10::weak_intrusive_ptr<c10::StorageImpl> storage;
  const void *storage_raw;
  int64_t offset, numel, E;
  uint32_t version;
  at::Tensor row_index;
};
std::list<CsrEntry> g_csr;

at::Tensor csr_row_index(const at::Tensor &indptr, int64_t E) {
  c10::StorageImpl *raw = indptr.storage().unsafeGetStorageImpl();
  const uint32_t ver = version_of(indptr);
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto it = g_csr.begin(); it != g_csr.end();) {
      if (it->storage.expired()) {          // the indptr tensor is gone: drop its [E] row index (8 bytes per edge)
        it = g_csr.erase(it);
        continue;
      }
      if (it->storage_raw == raw && it->offset == indptr.storage_offset() && it->numel == indptr.numel() && it->E == E &&
          it->version == ver) {
        g_csr.splice(g_csr.begin(), g_csr, it);
        return it->row_index;
      }
      ++it;
    }
  }
  at::Tensor row = at::empty({E}, indptr.options().dtype(at::kLong));
  check_status(geot_b200_csr_to_coo(indptr.data_ptr(), indptr.scalar_type() == at::kLong ? 64 : 32, indptr.numel() - 1, E,
                                    row.data_ptr<int64_t>(), at::cuda::getCurrentCUDAStream()),
               "csr_to_coo");
  CsrEntry e(indptr.storage().getWeakStorageImpl());
  e.storage_raw = raw; e.offset = indptr.storage_offset(); e.numel = indptr.numel(); e.E = E; e.version = ver; e.row_index = row;
  std::lock_guard<std::mutex> lk(g_plan_mu);
  g_csr.push_front(std::move(e));
  while (g_csr.size() > 4) g_csr.pop_back();      // an entry holds 8 bytes per edge: keep few
  return row;
}

void clear_csr_cache() {
  std::lock_guard<std::mutex> lk(g_plan_mu);
  g_csr.clear();
}

// geot::csr_gws_impl -- csrc/csr_gws.cpp:24-35 + csrc/cuda/csr_gws_cuda.cu: out[r] = sum_{e in row r} weight[e] * src[indices[e]].
// Like the reference the output has indptr.size(0) rows (= nrow + 1, csr_gws.cpp:29-31); the last one is 0.
// The row index is expanded from indptr once per graph (cached) and the COO kernels do the rest.
at::Tensor csr_gws_impl(at::Tensor indptr, at::Tensor indices, at::Tensor weight, at::Tensor src) {
  TORCH_CHECK(src.is_cuda(), "geot::csr_gws: src must be a CUDA tensor (this build has no CPU path)");
  TORCH_CHECK(indptr.dim() == 1 && indices.dim() == 1 && indptr.numel() >= 2, "indptr and indices must be 1 dimensional");
  TORCH_CHECK(src.dim() == 2, "src must be 2 dimensional");
  TORCH_CHECK(weight.dim() == 1 && weight.numel() == indices.numel(), "weight must be 1 dimensional with one entry per nonzero");
  TORCH_CHECK(indptr.scalar_type() == at::kLong || indptr.scalar_type() == at::kInt, "indptr must be int32 or int64");
  TORCH_CHECK(indptr.is_cuda() && indptr.device() == src.device() && indices.is_cuda() && indices.device() == src.device(),
              "geot::csr_gws: indptr, indices and src must be on the same CUDA device");
  c10::cuda::CUDAGuard guard(src.device());
  const at::Tensor ptr = indptr.contiguous();
  const int64_t E = indices.numel(), nrow = ptr.numel() - 1;
  auto shape = src.sizes().vec();
  shape[0] = nrow + 1;
  if (E == 0) return at::zeros(shape, src.options());
  const at::Tensor row = csr_row_index(ptr, E);
  const at::Tensor col = indices.scalar_type() == at::kLong ? indices : indices.to(at::kLong);
  // rows after the last non-empty one (at least the reference's extra row) are 0
  return run("csr_gws", src, col, row, weight, 1, src.size(1), GEOT_SUM, GEOT_W_EDGE, true, src.sizes().vec(), nrow + 1);
}

// geot::coo_to_csr_impl -- geot/match_replace/format_transform.py:5-18: int32 rowptr [nrow+1], nrow = coo_row.max()+1.
at::Tensor coo_to_csr_impl(at::Tensor coo_row) {
  TORCH_CHECK(coo_row.is_cuda(), "geot::coo_to_csr: coo_row must be a CUDA tensor");
  TORCH_CHECK(coo_row.dim() == 1 && coo_row.numel() > 0, "coo_row must be 1 dimensional and non-empty");
  c10::cuda::CUDAGuard guard(coo_row.device());
  at::Tensor idx = (coo_row.scalar_type() == at::kLong ? coo_row : coo_row.to(at::kLong)).contiguous();
  at::Tensor buf;
  geot_plan_t plan = get_plan(idx, &buf);
  TORCH_CHECK(plan.is_sorted, "geot::coo_to_csr: coo_row is not sorted");
  at::Tensor rowptr = at::from_blob(const_cast<int64_t *>(plan.rowptr), {plan.S + 1}, [buf](void *) mutable { buf.reset(); },
                                    idx.options());
  return rowptr.to(at::kInt);
}

}  // namespace

TORCH_LIBRARY_FRAGMENT(geot, m) {
  // reference schemas
  m.def("index_scatter(int dim, Tensor index, Tensor src, str reduce, bool sorted) -> Tensor");
  m.def("gather_scatter_impl(Tensor src_index, Tensor dst_index, Tensor src) -> Tensor");
  m.def("gather_weight_scatter_impl(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src) -> Tensor");
  m.def("mh_spmm(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src, str reduce) -> Tensor");
  m.def("sddmm_coo_impl(Tensor src_index, Tensor dst_index, Tensor mat_1, Tensor mat_2) -> Tensor");
  m.def("csr_gws_impl(Tensor indptr, Tensor indices, Tensor weight, Tensor src) -> Tensor");
  m.def("coo_to_csr_impl(Tensor coo_row) -> Tensor");
  // additions: reduce-aware gather ops, the plan, the multi-GPU partition
  m.def("gather_scatter_reduce(Tensor src_index, Tensor dst_index, Tensor src, str reduce) -> Tensor");
  m.def("gather_weight_scatter_reduce(Tensor src_index, Tensor dst_index, Tensor weight, Tensor src, str reduce) -> Tensor");
  m.def("format_preprocess(Tensor dst_index) -> (Tensor, Tensor)");
  m.def("plan_shards(Tensor dst_index, int parts) -> Tensor");
  m.def("sddmm_mh_impl(Tensor src_index, Tensor dst_index, Tensor mat_1, Tensor mat_2, bool head_major) -> Tensor");
  m.def("segment_softmax(Tensor src, Tensor index) -> Tensor");
  m.def("segment_softmax_backward(Tensor out, Tensor grad_out, Tensor index) -> Tensor");
  m.def("gatv2_score(Tensor x_l, Tensor x_r, Tensor att, Tensor src_index, Tensor dst_index, float negative_slope) -> Tensor");
  m.def("gatv2_score_backward(Tensor grad, Tensor x_l, Tensor x_r, Tensor att, Tensor src_index, Tensor dst_index, "
        "Tensor t_perm, Tensor t_dst_index, Tensor t_src_index, float negative_slope, bool need_x_l, bool need_x_r, "
        "bool need_att) -> (Tensor, Tensor, Tensor)");
  m.def("graph_attention(Tensor q, Tensor k, Tensor v, Tensor src_index, Tensor dst_index, float scale) -> (Tensor, Tensor)");
  m.def("graph_attention_backward(Tensor grad, Tensor q, Tensor k, Tensor v, Tensor out, Tensor lse, Tensor src_index, "
        "Tensor dst_index, float scale) -> (Tensor, Tensor, Tensor)");
  m.def("clear_plan_cache() -> ()", []() { clear_plan_cache(); });
  m.def("abi_version() -> int", []() { return (int64_t)geot_b200_version(); });
}

TORCH_LIBRARY_IMPL(geot, CUDA, m) {
  m.impl("index_scatter", index_scatter_cuda_impl);
  m.impl("gather_scatter_impl", gather_scatter_impl);
  m.impl("gather_weight_scatter_impl", gather_weight_scatter_impl);
  m.impl("mh_spmm", mh_spmm_impl);
  m.impl("sddmm_coo_impl", sddmm_coo_impl);
  m.impl("csr_gws_impl", csr_gws_impl);
  m.impl("coo_to_csr_impl", coo_to_csr_impl);
  m.impl("gather_scatter_reduce", gather_scatter_reduce);
  m.impl("gather_weight_scatter_reduce", gather_weight_scatter_reduce);
  m.impl("format_preprocess", format_preprocess);
  m.impl("plan_shards", plan_shards);
  m.impl("sddmm_mh_impl", sddmm_mh_impl);
  m.impl("segment_softmax", segment_softmax_impl);
  m.impl("segment_softmax_backward", segment_softmax_backward_impl);
  m.impl("gatv2_score", gatv2_score_impl);
  m.impl("gatv2_score_backward", gatv2_score_backward_impl);
  m.impl("graph_attention", graph_attention_impl);
  m.impl("graph_attention_backward", graph_attention_backward_impl);
}
