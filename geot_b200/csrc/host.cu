// host.cu -- the host-buffer entries of the C ABI (include/geot_b200.h): the stateless geot_b200_segment_reduce_host
// and the resident host graph (geot_b200_host_graph_*).  Both run one pipeline: src first, then the sorted edge list
// in slices cut at segment boundaries.  Slice k+1 is copied (H2D stream) while slice k is reduced (compute stream)
// and the finished dst rows of slice k-1 travel back (D2H stream, the other direction of the link).  No kernel of
// its own: the slices go through segment_reduce_impl (abi.cu).
#include <cuda_runtime.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "internal.h"

namespace {

constexpr int kMaxSlices = 64;

int default_host_threads() { return (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency())); }

// fn(begin, end) over [0, n) on up to `threads` host threads (the calling thread takes the first share)
template <typename F>
void parallel_ranges(int threads, int64_t n, F fn) {
  if (n <= 0) return;
  threads = (int)std::max<int64_t>(1, std::min<int64_t>(threads, n / 4096 + 1));
  if (threads == 1) { fn((int64_t)0, n); return; }
  std::vector<std::thread> pool;
  const int64_t per = (n + threads - 1) / threads;
  for (int t = 1; t < threads; ++t) {
    const int64_t b = per * t, e = std::min(n, b + per);
    if (b < e) pool.emplace_back([=] { fn(b, e); });
  }
  fn((int64_t)0, std::min(n, per));
  for (auto &th : pool) th.join();
}

// rp[i] = first position in idx[0, n) whose value is >= row0 + i, for i in [0, rows]  (idx sorted): the slice's CSR
// row pointer.  Rows are walked in order, galloping from the previous boundary, so the cost follows the number of
// cache lines a row spans rather than log2(n) misses per row.
void host_row_pointers(const int64_t *idx, int64_t n, int64_t row0, int64_t rows, int64_t *rp, int threads) {
  parallel_ranges(threads, rows + 1, [=](int64_t ia, int64_t ib) {
    int64_t pos = std::lower_bound(idx, idx + n, row0 + ia) - idx;
    for (int64_t i = ia; i < ib; ++i) {
      const int64_t target = row0 + i;
      if (pos < n && idx[pos] < target) {
        int64_t lo = pos, step = 1;
        while (lo + step < n && idx[lo + step] < target) { lo += step; step <<= 1; }
        const int64_t hi = std::min(n, lo + step);
        pos = std::lower_bound(idx + lo + 1, idx + hi, target) - idx;
      }
      rp[i] = pos;
    }
  });
}

// Cuts the sorted edge list [0, E) into at most `want` slices of about E / want edges, each cut moved right to a
// segment boundary: slice k is edges [cut[k], cut[k+1]) and owns dst rows [row[k], row[k+1]), row[0] = 0 and
// row[n] = S.  Returns n, or 0 when the index is invalid.  Only dst_index[0], the cuts and dst_index[E-1] are
// checked: read in that order they must be non-decreasing and in [0, S), so that every row range lies in [0, S) and
// the D2H copies sized from them stay inside dst.  Checking the whole index would cost a pass over E; the rest of
// it is trusted to be sorted, as on the device path.
int cut_at_segments(const int64_t *di, int64_t E, int64_t S, int want, int64_t *cut, int64_t *row) {
  if (di[0] < 0 || di[E - 1] >= S) return 0;
  cut[0] = 0;
  row[0] = 0;
  int n = 0;
  for (int k = 1; k <= want; ++k) {
    int64_t c = (k == want) ? E : (E / want) * k;
    while (c < E && c > 0 && di[c] == di[c - 1]) ++c;   // move right to a segment boundary
    if (c > cut[n]) {
      if (c < E && (di[c] < di[cut[n]] || di[c] > di[E - 1])) return 0;
      ++n;
      cut[n] = c;
      row[n] = (c < E) ? di[c] : S;
    }
    if (c >= E) break;
  }
  return n;
}

// The slices of one call (at most kMaxSlices, cut as above).
struct Slices {
  int n = 0;
  int64_t cut[kMaxSlices + 1];
  int64_t row[kMaxSlices + 1];
  int64_t max_edges() const {
    int64_t m = 0;
    for (int k = 0; k < n; ++k) m = std::max(m, cut[k + 1] - cut[k]);
    return m;
  }
};

// Device buffers of one call: src, dst, two staging halves for the slices' operands, the reduction's workspace.
struct Buffers {
  char *src, *dst, *half[2];
  void *ws;
};

// The streams, events and device memory of one pipeline, all on device `dev`.
struct Pipeline {
  int dev = -1;
  cudaStream_t h2d = nullptr, comp = nullptr, d2h = nullptr;
  cudaEvent_t copied[kMaxSlices] = {}, reduced[kMaxSlices] = {};
  cudaEvent_t src_ready = nullptr;
  char *resident = nullptr;       // allocated once by init: a host graph's index arrays
  char *buf = nullptr;            // the per-call Buffers, grown on demand and reused across calls
  size_t buf_bytes = 0;
  unsigned long long last_h2d = 0, last_d2h = 0;   // bytes the last call moved over the link

  // On the current device.  After a failure the caller releases what was created.
  int init(size_t resident_bytes) {
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&comp, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&d2h, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&src_ready, cudaEventDisableTiming));
    for (int i = 0; i < kMaxSlices; ++i) {
      CUDA_TRY(cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&reduced[i], cudaEventDisableTiming));
    }
    if (resident_bytes) CUDA_TRY(cudaMalloc(&resident, resident_bytes));
    return GEOT_OK;
  }

  // Frees everything on `dev`; the caller's current device stays current.
  void release() {
    int cur = 0;
    const bool switch_dev = dev >= 0 && cudaGetDevice(&cur) == cudaSuccess;
    if (switch_dev) cudaSetDevice(dev);
    if (resident) cudaFree(resident);
    if (buf) cudaFree(buf);
    for (int i = 0; i < kMaxSlices; ++i) {
      if (copied[i]) cudaEventDestroy(copied[i]);
      if (reduced[i]) cudaEventDestroy(reduced[i]);
    }
    if (src_ready) cudaEventDestroy(src_ready);
    if (h2d) cudaStreamDestroy(h2d);
    if (comp) cudaStreamDestroy(comp);
    if (d2h) cudaStreamDestroy(d2h);
    if (switch_dev) cudaSetDevice(cur);
    *this = Pipeline();
  }

  int buffers(size_t b_src, size_t b_dst, size_t half_bytes, size_t b_ws, Buffers *b) {
    const size_t total = align256(b_src) + align256(b_dst) + 2 * half_bytes + align256(b_ws);
    if (buf_bytes < total) {
      if (buf) CUDA_TRY(cudaFree(buf));
      buf = nullptr; buf_bytes = 0;
      CUDA_TRY(cudaMalloc(&buf, total));
      buf_bytes = total;
    }
    char *p = buf;
    b->src = p; p += align256(b_src);
    b->dst = p; p += align256(b_dst);
    b->half[0] = p; b->half[1] = p + half_bytes; p += 2 * half_bytes;
    b->ws = p;
    return GEOT_OK;
  }
};

// Runs the slices through the pipeline.  The caller has enqueued src on pp.h2d (h2d_bytes so far) and whatever
// pp.comp must do first.  Per slice k: upload(k, half, h2d_bytes) enqueues its operands into staging half `half` on
// pp.h2d and adds the bytes it moved; reduce(k, half) enqueues its reduction into d_dst on pp.comp.  Returns when
// rows [row[0], row[n]) of d_dst are in dst (host).
template <typename Upload, typename Reduce>
int run_slices(Pipeline &pp, const Slices &s, unsigned long long h2d_bytes, size_t row_bytes, const char *d_dst,
               void *dst, Upload upload, Reduce reduce) {
  CUDA_TRY(cudaEventRecord(pp.src_ready, pp.h2d));
  CUDA_TRY(cudaStreamWaitEvent(pp.comp, pp.src_ready, 0));
  unsigned long long d2h_bytes = 0;
  for (int k = 0; k < s.n; ++k) {
    if (k >= 2) CUDA_TRY(cudaStreamWaitEvent(pp.h2d, pp.reduced[k - 2], 0));   // half k & 1 is free once slice k-2 is reduced
    if (int rc = upload(k, k & 1, h2d_bytes); rc != GEOT_OK) return rc;
    CUDA_TRY(cudaEventRecord(pp.copied[k], pp.h2d));
    CUDA_TRY(cudaStreamWaitEvent(pp.comp, pp.copied[k], 0));
    if (int rc = reduce(k, k & 1); rc != GEOT_OK) { cudaDeviceSynchronize(); return rc; }
    CUDA_TRY(cudaEventRecord(pp.reduced[k], pp.comp));
    // rows [row[k], row[k+1]) are final: send them home
    CUDA_TRY(cudaStreamWaitEvent(pp.d2h, pp.reduced[k], 0));
    const size_t off = (size_t)s.row[k] * row_bytes, bytes = (size_t)(s.row[k + 1] - s.row[k]) * row_bytes;
    CUDA_TRY(cudaMemcpyAsync(static_cast<char *>(dst) + off, d_dst + off, bytes, cudaMemcpyDeviceToHost, pp.d2h));
    d2h_bytes += bytes;
  }
  CUDA_TRY(cudaStreamSynchronize(pp.d2h));
  CUDA_TRY(cudaStreamSynchronize(pp.comp));
  CUDA_TRY(cudaStreamSynchronize(pp.h2d));
  pp.last_h2d = h2d_bytes;
  pp.last_d2h = d2h_bytes;
  return GEOT_OK;
}

// The stateless entry's per-process pipeline, and the pinned host staging of the row-pointer transport.
struct Arena {
  Pipeline pp;
  char *pinned = nullptr;         // double-buffered: the row pointers of slices k and k+1
  size_t pinned_bytes = 0;
};
Arena g_arena;

}  // namespace

struct geot_host_graph {
  int64_t E = 0, S = 0, N_src = 0;
  bool gather = false;
  int64_t *d_di = nullptr, *d_si = nullptr;     // resident indices (in pp.resident)
  static constexpr int kFine = 256;             // fine cuts at segment boundaries; a call groups them into slices
  int n_fine = 0;
  int64_t cut[kFine + 1];                       // edge offsets
  int64_t row_cut[kFine + 1];                   // first dst row of every fine slice (row_cut[0] = 0, row_cut[n_fine] = S)
  Pipeline pp;
};

extern "C" {

// ---- stateless host-buffer entry ----------------------------------------------------------------------

int geot_b200_host_arena_release(void) {
  Arena &a = g_arena;
  a.pp.release();
  if (a.pinned) cudaFreeHost(a.pinned);
  a = Arena();
  return GEOT_OK;
}

int geot_b200_segment_reduce_host(const void *src, int64_t N_src, const int64_t *src_index,
                                  const int64_t *dst_index, const void *weight, void *dst, int64_t E, int64_t S,
                                  int64_t H, int64_t F, int dtype, int reduce, int weight_layout) {
  if (!src || !dst_index || !dst || N_src <= 0) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  if (S <= 0 || H <= 0 || F <= 0 || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if ((weight_layout == GEOT_W_NONE) != (weight == nullptr)) return GEOT_ERR_INVALID_ARG;
  if (weight_layout == GEOT_W_HEAD_EDGE && H > 1) return GEOT_ERR_UNSUPPORTED;  // [H,E] cannot be sliced by edge
  const int64_t W = H * F;
  const size_t es = dtype_size(dtype);
  const size_t wpe = weight ? (weight_layout == GEOT_W_EDGE ? 1 : (size_t)H) * es : 0;   // weight bytes per edge
  const bool gather = src_index != nullptr;
  const size_t b_src = (gather ? (size_t)N_src : 0) * W * es;   // index_scatter: src rows are edge-aligned, sliced
  const size_t src_pe = gather ? 0 : (size_t)W * es;            // src bytes per edge when sliced
  const size_t b_dst = (size_t)S * W * es;

  // slices: about 128 MB of edge-aligned operands each, at least 4, cut at segment boundaries
  const size_t per_edge = 8 + (gather ? 8 : 0) + wpe + src_pe;
  int want = (int)std::min<size_t>(kMaxSlices, std::max<size_t>(4, ((size_t)E * per_edge) >> 27));
  if (E < 4096) want = 1;
  Slices s;
  s.n = cut_at_segments(dst_index, E, S, want, s.cut, s.row);
  if (s.n == 0) return GEOT_ERR_INVALID_ARG;
  const int64_t max_slice = s.max_edges();

  // Row-pointer transport (default; GEOT_B200_HOST_COMPACT=0 turns it off): each slice sends its CSR row pointer
  // (rows + 1 values, computed on the host threads while the previous slice is on the link) instead of its dst_index
  // (one value per edge) and the device expands it.  Same results bit for bit; Reddit-shape gws moves 1.49 GB
  // instead of 2.41 GB per call: 44.5 -> 28.1 ms (profiles/r02a_bench_compact*.json).  Narrowing src_index to int32
  // on the host was measured too and lost (37.2 ms: the host pass costs more than the bytes it saves) -- removed.
  const bool c_rows = env_int("GEOT_B200_HOST_COMPACT", 1) != 0;
  int host_threads = env_int("GEOT_B200_HOST_THREADS", 0);
  if (host_threads <= 0) host_threads = default_host_threads();
  int64_t max_rows = 0;
  for (int k = 0; k < s.n; ++k) max_rows = std::max(max_rows, s.row[k + 1] - s.row[k]);
  const size_t stage_rp = c_rows ? align256((size_t)(max_rows + 1) * 8) : 0;

  // a staging half: dst ids (expanded from the row pointer, or as given), src ids, weights, edge-aligned src rows,
  // row pointer
  const size_t a_id = align256((size_t)max_slice * 8), a_w = align256((size_t)max_slice * wpe);
  const size_t a_x = align256((size_t)max_slice * src_pe);
  const size_t b_ws = geot_b200_workspace_bytes(max_slice, W, dtype, 1);
  Arena &a = g_arena;
  int cur_dev = 0;
  CUDA_TRY(cudaGetDevice(&cur_dev));
  if (a.pp.dev != cur_dev) {      // first call, or the arena belongs to another device: start over on this one
    geot_b200_host_arena_release();
    if (int rc = a.pp.init(0); rc != GEOT_OK) { geot_b200_host_arena_release(); return rc; }
  }
  Buffers b;
  if (int rc = a.pp.buffers(b_src, b_dst, a_id * (gather ? 2 : 1) + a_w + a_x + stage_rp, b_ws, &b); rc != GEOT_OK) return rc;
  if (a.pinned_bytes < 2 * stage_rp) {
    if (a.pinned) CUDA_TRY(cudaFreeHost(a.pinned));
    a.pinned = nullptr; a.pinned_bytes = 0;
    CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&a.pinned), 2 * stage_rp, cudaHostAllocDefault));
    a.pinned_bytes = 2 * stage_rp;
  }
  struct Stage { int64_t *di, *si, *rp; char *w, *x; } st[2];
  for (int h = 0; h < 2; ++h) {
    char *q = b.half[h];
    st[h].di = reinterpret_cast<int64_t *>(q); q += a_id;
    st[h].si = gather ? reinterpret_cast<int64_t *>(q) : nullptr; q += gather ? a_id : 0;
    st[h].w = q; q += a_w;
    st[h].x = q; q += a_x;
    st[h].rp = reinterpret_cast<int64_t *>(q);
  }

  CUDA_TRY(cudaMemsetAsync(b.dst, 0, b_dst, a.pp.comp));      // empty rows read 0; slices never clear
  if (gather) CUDA_TRY(cudaMemcpyAsync(b.src, src, b_src, cudaMemcpyHostToDevice, a.pp.h2d));
  auto upload = [&](int k, int h, unsigned long long &bytes) -> int {
    const int64_t e0 = s.cut[k], n = s.cut[k + 1] - e0, rows = s.row[k + 1] - s.row[k];
    if (c_rows) {
      // the host threads prepare slice k while slice k-1 is on the link; the pinned half is free once the copies of
      // slice k-2 have left it
      int64_t *h_rp = reinterpret_cast<int64_t *>(a.pinned + (size_t)h * stage_rp);
      if (k >= 2) CUDA_TRY(cudaEventSynchronize(a.pp.copied[k - 2]));
      host_row_pointers(dst_index + e0, n, s.row[k], rows, h_rp, host_threads);
      CUDA_TRY(cudaMemcpyAsync(st[h].rp, h_rp, (size_t)(rows + 1) * 8, cudaMemcpyHostToDevice, a.pp.h2d));
      bytes += (size_t)(rows + 1) * 8;
    } else {
      CUDA_TRY(cudaMemcpyAsync(st[h].di, dst_index + e0, (size_t)n * 8, cudaMemcpyHostToDevice, a.pp.h2d));
      bytes += (size_t)n * 8;
    }
    if (gather) {
      CUDA_TRY(cudaMemcpyAsync(st[h].si, src_index + e0, (size_t)n * 8, cudaMemcpyHostToDevice, a.pp.h2d));
      bytes += (size_t)n * 8;
    }
    if (weight) CUDA_TRY(cudaMemcpyAsync(st[h].w, static_cast<const char *>(weight) + (size_t)e0 * wpe, (size_t)n * wpe, cudaMemcpyHostToDevice, a.pp.h2d));
    if (!gather) CUDA_TRY(cudaMemcpyAsync(st[h].x, static_cast<const char *>(src) + (size_t)e0 * src_pe, (size_t)n * src_pe, cudaMemcpyHostToDevice, a.pp.h2d));
    bytes += (size_t)n * (wpe + src_pe);
    return GEOT_OK;
  };
  Extra never_clear;
  never_clear.clear_mode = 1;
  auto reduce_slice = [&](int k, int h) -> int {
    const int64_t n = s.cut[k + 1] - s.cut[k], r0 = s.row[k], rows = s.row[k + 1] - r0;
    const void *x = gather ? b.src : st[h].x;
    const void *w = weight ? st[h].w : nullptr;
    if (!c_rows)
      return segment_reduce_impl(x, st[h].si, st[h].di, w, b.dst, n, S, H, F, dtype, reduce, weight_layout, 1, nullptr,
                                 b.ws, b_ws, a.pp.comp, nullptr, never_clear);
    // expand the row pointer into slice-local dst ids [0, rows): the slice's rows start at d_dst + r0 * W
    if (int rc = geot_b200_csr_to_coo(st[h].rp, 64, rows, n, st[h].di, a.pp.comp); rc != GEOT_OK) return rc;
    return segment_reduce_impl(x, st[h].si, st[h].di, w, b.dst + (size_t)r0 * W * es, n, rows, H, F, dtype, reduce,
                               weight_layout, 1, nullptr, b.ws, b_ws, a.pp.comp, nullptr, never_clear);
  };
  return run_slices(a.pp, s, gather ? b_src : 0, (size_t)W * es, b.dst, dst, upload, reduce_slice);
}

int geot_b200_host_last_transfer(unsigned long long *h2d_bytes, unsigned long long *d2h_bytes) {
  if (h2d_bytes) *h2d_bytes = g_arena.pp.last_h2d;
  if (d2h_bytes) *d2h_bytes = g_arena.pp.last_d2h;
  return GEOT_OK;
}

int geot_b200_host_row_pointers(const int64_t *index, int64_t n, int64_t row0, int64_t rows, int64_t *rowptr, int threads) {
  if (!index || !rowptr || n < 0 || rows < 0) return GEOT_ERR_INVALID_ARG;
  if (threads <= 0) threads = default_host_threads();
  host_row_pointers(index, n, row0, rows, rowptr, threads);
  return GEOT_OK;
}

// ---- resident host graph -------------------------------------------------------------------------------
// The graph (index arrays) of a GNN is static across layers and epochs while the features and edge weights change
// every call.  A host graph handle uploads the indices ONCE; every reduce call then ships only src (+ weights) over
// the link and brings dst back: Reddit-shape gather_weight_scatter moves 0.58 GB per call instead of 2.41 GB.
int geot_b200_host_graph_destroy(geot_host_graph_t *g) {
  if (!g) return GEOT_OK;
  g->pp.release();
  delete g;
  return GEOT_OK;
}

int geot_b200_host_graph_create(const int64_t *src_index, const int64_t *dst_index, int64_t E, int64_t S, int64_t N_src,
                                geot_host_graph_t **out) {
  if (!dst_index || !out || S <= 0 || (src_index && N_src <= 0)) return GEOT_ERR_INVALID_ARG;
  if (E <= 0) return GEOT_ERR_EMPTY;
  geot_host_graph *g = new geot_host_graph();
  g->E = E; g->S = S; g->N_src = N_src; g->gather = src_index != nullptr;
  // fine cuts: about E / kFine edges each, moved right to a segment boundary
  const int want = (int)std::min<int64_t>(geot_host_graph::kFine, std::max<int64_t>(1, E / 65536));
  g->n_fine = cut_at_segments(dst_index, E, S, want, g->cut, g->row_cut);
  const size_t a_id = align256((size_t)E * 8);
  auto upload = [&]() -> int {
    if (int rc = g->pp.init(a_id * (g->gather ? 2 : 1)); rc != GEOT_OK) return rc;
    g->d_di = reinterpret_cast<int64_t *>(g->pp.resident);
    g->d_si = g->gather ? reinterpret_cast<int64_t *>(g->pp.resident + a_id) : nullptr;
    CUDA_TRY(cudaMemcpyAsync(g->d_di, dst_index, (size_t)E * 8, cudaMemcpyHostToDevice, g->pp.h2d));
    if (g->gather) CUDA_TRY(cudaMemcpyAsync(g->d_si, src_index, (size_t)E * 8, cudaMemcpyHostToDevice, g->pp.h2d));
    CUDA_TRY(cudaStreamSynchronize(g->pp.h2d));
    return GEOT_OK;
  };
  const int rc = g->n_fine == 0 ? GEOT_ERR_INVALID_ARG : upload();
  if (rc != GEOT_OK) { geot_b200_host_graph_destroy(g); return rc; }
  *out = g;
  return GEOT_OK;
}

int geot_b200_host_graph_reduce(geot_host_graph_t *g, const void *src, const void *weight, void *dst, int64_t H,
                                int64_t F, int dtype, int reduce, int weight_layout) {
  if (!g || !src || !dst) return GEOT_ERR_INVALID_ARG;
  if (H <= 0 || F <= 0 || dtype < GEOT_F32 || dtype > GEOT_F16) return GEOT_ERR_INVALID_ARG;
  if ((weight_layout == GEOT_W_NONE) != (weight == nullptr)) return GEOT_ERR_INVALID_ARG;
  if (weight_layout == GEOT_W_HEAD_EDGE && H > 1) return GEOT_ERR_UNSUPPORTED;  // [H,E] cannot be sliced by edge
  int cur_dev = 0;
  CUDA_TRY(cudaGetDevice(&cur_dev));
  if (cur_dev != g->pp.dev) return GEOT_ERR_INVALID_ARG;       // the handle lives on the device it was created on
  const int64_t E = g->E, S = g->S, W = H * F;
  const size_t es = dtype_size(dtype);
  const size_t wpe = weight ? (weight_layout == GEOT_W_EDGE ? 1 : (size_t)H) * es : 0;
  const size_t src_pe = g->gather ? 0 : (size_t)W * es;
  const size_t b_src = g->gather ? (size_t)g->N_src * W * es : 0;
  const size_t b_dst = (size_t)S * W * es;

  // group the fine cuts into slices of about 48 MB of per-edge payload (at least 4 when the graph allows, at most 64)
  const size_t per_edge = std::max<size_t>(wpe + src_pe, 1);
  int n_slices = (int)std::min<size_t>(kMaxSlices, std::max<size_t>(4, ((size_t)E * per_edge) / (48u << 20)));
  n_slices = std::min(n_slices, g->n_fine);
  Slices s;
  s.n = n_slices;
  for (int k = 0; k <= n_slices; ++k) {
    const int f = (int)(((int64_t)g->n_fine * k) / n_slices);
    s.cut[k] = g->cut[f];
    s.row[k] = g->row_cut[f];
  }
  const int64_t max_slice = s.max_edges();

  // a staging half: weights, edge-aligned src rows
  const size_t a_w = align256((size_t)max_slice * wpe), a_x = align256((size_t)max_slice * src_pe);
  const size_t b_ws = geot_b200_workspace_bytes(max_slice, W, dtype, 1);
  Buffers b;
  if (int rc = g->pp.buffers(b_src, b_dst, a_w + a_x, b_ws, &b); rc != GEOT_OK) return rc;

  if (g->gather) CUDA_TRY(cudaMemcpyAsync(b.src, src, b_src, cudaMemcpyHostToDevice, g->pp.h2d));
  auto upload = [&](int k, int h, unsigned long long &bytes) -> int {
    const int64_t e0 = s.cut[k], n = s.cut[k + 1] - e0;
    if (weight) CUDA_TRY(cudaMemcpyAsync(b.half[h], static_cast<const char *>(weight) + (size_t)e0 * wpe, (size_t)n * wpe, cudaMemcpyHostToDevice, g->pp.h2d));
    if (!g->gather) CUDA_TRY(cudaMemcpyAsync(b.half[h] + a_w, static_cast<const char *>(src) + (size_t)e0 * src_pe, (size_t)n * src_pe, cudaMemcpyHostToDevice, g->pp.h2d));
    bytes += (size_t)n * (wpe + src_pe);
    return GEOT_OK;
  };
  auto reduce_slice = [&](int k, int h) -> int {
    const int64_t e0 = s.cut[k], n = s.cut[k + 1] - e0;
    Extra ex;                      // rows without edges inside [row[k], row[k+1]) are zero-filled by the kernel: no memset
    ex.fill_lo = s.row[k];
    ex.fill_hi = s.row[k + 1];
    return segment_reduce_impl(g->gather ? b.src : b.half[h] + a_w, g->gather ? g->d_si + e0 : nullptr, g->d_di + e0,
                               weight ? b.half[h] : nullptr, b.dst, n, S, H, F, dtype, reduce, weight_layout, 1, nullptr,
                               b.ws, b_ws, g->pp.comp, nullptr, ex);
  };
  return run_slices(g->pp, s, b_src, (size_t)W * es, b.dst, dst, upload, reduce_slice);
}

int geot_b200_host_graph_last_transfer(const geot_host_graph_t *g, unsigned long long *h2d_bytes, unsigned long long *d2h_bytes,
                                       unsigned long long *resident_bytes) {
  if (!g) return GEOT_ERR_INVALID_ARG;
  if (h2d_bytes) *h2d_bytes = g->pp.last_h2d;
  if (d2h_bytes) *d2h_bytes = g->pp.last_d2h;
  if (resident_bytes) *resident_bytes = (unsigned long long)g->E * 8 * (g->gather ? 2 : 1);
  return GEOT_OK;
}

}  // extern "C"
