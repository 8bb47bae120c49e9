// extern "C" boundary (include/scn_b200.h).  No torch types: raw device pointers, sizes, a stream.
#include "../../include/scn_b200.h"
#include "metadata.cuh"
#include <algorithm>
#include <atomic>
#include <mutex>
#include <thread>
#include <vector>
#include <map>
#include <deque>
#include <condition_variable>
#include <chrono>
#include <stdlib.h>

namespace scn {
std::atomic<long> g_launches{0};
std::atomic<long> g_counters[kCntCounters];
void epilogue_stats_arm(double *sums);
bool epilogue_stats_take();
void lateral_arm(const float *in, const void *in16, const float *w, long long tag, int Cin, long rows);
bool lateral_take();
namespace {
struct TlEv { const char *who; int kind; long a, b; double t; };
std::vector<TlEv> g_tl;
std::mutex g_tl_mu;
int g_tl_on = -1;
double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
} // namespace
int pdl_mode() {
  static int on = -1;
  if (on < 0) on = getenv("SCN_PDL") ? atoi(getenv("SCN_PDL")) : 0;
  return on;
}
void timeline_mark(const char *who, int kind, long a, long b) {
  if (g_tl_on < 0) g_tl_on = getenv("SCN_TIMELINE") ? atoi(getenv("SCN_TIMELINE")) : 0;
  if (!g_tl_on) return;
  std::lock_guard<std::mutex> lk(g_tl_mu);
  g_tl.push_back(TlEv{who, kind, a, b, now_us()});
}
void timeline_dump() {
  if (g_tl_on <= 0) return;
  std::lock_guard<std::mutex> lk(g_tl_mu);
  if (g_tl.empty()) return;
  const double t0 = g_tl[0].t;
  for (const TlEv &e : g_tl) fprintf(stderr, "[tl] %8.1f us %-8s kind %d  %ld %ld\n", e.t - t0, e.who, e.kind, e.a, e.b);
  g_tl.clear();
}
const char *last_error();
void set_prefetch_worker_thread(bool on, int ctx);
int launch_conv_plan_simt(const float *in, float *out, const float *W, const int *nbr, const int *outRow, int nOut, int K, int Cin, int Cout,
                          const float *bias, cudaStream_t s);
int launch_conv_list_simt(const float *in, float *out, const float *W, const int2 *pairs, const int *d_off, const int *offHost, int K, int Cin,
                          int Cout, int srcIsY, int singlePass, cudaStream_t s);
int bn_forward(const float *x, float *y, long n, int C, float *saveMean, float *saveInvStd, float *runningMean, float *runningVar,
               const float *weight, const float *bias, float eps, float momentum, int mode, float leak, void *workspace, cudaStream_t s, void *y16);
int bn_backward(const float *x, float *dx, const float *y, float *dy, long n, int C, const float *saveMean, const float *saveInvStd,
                const float *weight, float *dWeight, float *dBias, float leak, void *workspace, cudaStream_t s, const void *y16 = nullptr);
int input_forward(const float *in, float *out, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s);
int input_forward_pad16(const float *in, float *out, void *out16, int nOut, int maxActive, int C, int Cp, const int *tab, int average, cudaStream_t s);
int input_backward(float *din, const float *dout, long nIn, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s);
int add_rows(const float *a, const float *b, float *o, long n, cudaStream_t s, void *o16);
int conv_backward_simt(const float *in, float *d_in, const float *d_out, const float *W, float *dW, float *d_bias, const int2 *pairs,
                       const int *d_off, const int *offHost, int K, long nInRows, long nOutRows, int Cin, int Cout, int srcIsY, cudaStream_t s, int skipDIn = 0, int mathMode = 0,
                       const void *in16 = nullptr, const void *dout16 = nullptr, const int *planNbr = nullptr, const int *planOutRow = nullptr,
                       const unsigned long long *planMask = nullptr, int planPos = 0);
int dout_bf16_copy(const float *d_out, long n, cudaStream_t s, const void **out);
bool dw_plan_ok(int Cin, int Cout, int K, int mathMode);
void bwd_in16_arm(const void *in16);
const void *bwd_in16_take();
int transpose_weights(const float *W, float *Wt, int K, int Cin, int Cout, int reverse, cudaStream_t s);
int tc_available();
void set_pool_growth(int on);
long debug_chunk_mallocs();
long debug_chunk_waits();
long debug_chunk_total_mb();
long release_idle_chunks();
long release_conv_caches();
int launch_conv_plan_tc(const float *in, float *out, const float *W, const int *nbr, const int *outRow, const unsigned long long *tileMask,
                        int nOut, int K, int Cin, int Cout, const float *bias, int mathMode, cudaStream_t s, const int *tileW, int nWeights,
                        long nInRows, const void *in16, long long wTag, const float *addend, void *out16, long nOutRows, int CinW = 0, int wT = 0);
int to_bf16(const float *x, void *y, long n, cudaStream_t s);
int dense_rows_dw(const float *in, const float *d_out, float *dW, float *d_bias, long n, int Cin, int Cout, cudaStream_t s);
static int g_math_mode = 0;
static std::atomic<int> g_deterministic{0};
bool deterministic() { return g_deterministic.load(std::memory_order_relaxed) != 0; }
} // namespace scn

// The caller's thread and the prefetch worker (scn_metadata_prefetch) build into the same lazily
// filled caches; Metadata::buildMu / mapMu (metadata.cuh) keep them apart.
struct PrefetchOp { long v[13]; }; // kind, a[3], b[3], f[3], s[3]
struct scn_metadata {
  scn::Metadata md;
  // prefetch jobs of this Metadata that the process-wide worker threads have not finished yet
  std::mutex jobMu;
  std::condition_variable jobCv;
  int pending = 0;
  std::atomic<bool> stop{false};
  std::vector<PrefetchOp> ops, ops2; // chain worker (strided convolutions = the grid pyramid) / everything else
  // input-layer arguments of a job that starts with the input layer itself (kind 0, scn_metadata_build_reference_grids)
  long inSz[3] = {0, 0, 0}; const long *inCoords = nullptr; int inOnDevice = 0; long inRows = 0; int inCols = 0, inBatch = 0, inMode = 0;
  int device = 0;
  std::map<scn::P3, scn::RuleBookDev> s2d; // SparseToDense rulebooks (parity / inspection only: the scatter kernel does not need them)
};

using scn::Metadata;
namespace scn {
Metadata *metadata_of(scn_metadata *m) { return &m->md; }
int build_subm_on_caller(Metadata &md, const long *sz, const long *f);
int build_subm_on_caller(scn_metadata *m, const long *sz, const long *f) { return m ? build_subm_on_caller(m->md, sz, f) : -3; }
} // for the translation units that only see the opaque handle

#define M_OR_FAIL(m)                               \
  if (!(m)) {                                      \
    scn::set_error("null scn_metadata handle");    \
    return -3;                                     \
  }


extern "C" {

const char *scn_last_error(void) { return scn::last_error(); }
int scn_version(void) { return 1; }
int scn_n_rulebook_bits(void) { return 32; }
long scn_kernel_launch_count(void) { return scn::g_launches; }
int scn_set_pool_growth(int on) { scn::set_pool_growth(on); return 0; }
long scn_debug_counter(int which) {
  if (which >= 3 && which < scn::kCntCounters) return scn::g_counters[which].load();
  return which == 0 ? scn::debug_chunk_mallocs() : which == 1 ? scn::debug_chunk_waits() : scn::debug_chunk_total_mb();
}
long scn_release_cached_memory(void) {
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  return scn::release_idle_chunks() + scn::release_conv_caches();
}
int scn_fuse_next_lateral(const float *lat_in, const void *lat_in_bf16, const float *lat_weight, long long weight_tag, int n_in, long rows) {
  SCN_CHECK(lat_in && lat_weight && n_in > 0 && rows >= 0, "lateral request");
  scn::lateral_arm(lat_in, lat_in_bf16, lat_weight, weight_tag, n_in, rows);
  return 0;
}
int scn_fuse_next_stats(double *sums) {
  SCN_CHECK(sums, "statistics buffer");
  scn::epilogue_stats_arm(sums);
  return 0;
}
int scn_fuse_result(int *lateral_taken, int *stats_taken) {
  const bool l = scn::lateral_take(), st = scn::epilogue_stats_take();
  if (lateral_taken) *lateral_taken = l ? 1 : 0;
  if (stats_taken) *stats_taken = st ? 1 : 0;
  return 0;
}
int scn_set_math_mode(int mode) {
  if (mode < 0 || mode > 2) { scn::set_error("math mode must be 0 (fp32), 1 (tf32) or 2 (bf16)"); return -2; }
  scn::g_math_mode = mode;
  return 0;
}
int scn_get_math_mode(void) { return scn::g_math_mode; }
int scn_set_deterministic(int on) {
  scn::g_deterministic = on ? 1 : 0;
  return 0;
}
int scn_get_deterministic(void) { return scn::g_deterministic.load(); }
int scn_tensor_core_path_available(void) { return scn::tc_available(); }

int scn_metadata_create(scn_metadata **out, void *stream) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    scn::set_error("no CUDA device: this library has no CPU fallback");
    return -1;
  }
  scn_metadata *m = new scn_metadata();
  cudaGetDevice(&m->device);
  m->md.cstream = static_cast<cudaStream_t>(stream);
  int r = m->md.init();
  if (r) { delete m; return r; }
  *out = m;
  return 0;
}
static void wait_jobs(scn_metadata *m) {
  std::unique_lock<std::mutex> lk(m->jobMu);
  m->jobCv.wait(lk, [&] { return m->pending == 0; });
}
void scn_metadata_destroy(scn_metadata *m) {
  if (!m) return;
  m->stop = true;
  m->md.set_chain_done(true);
  wait_jobs(m);
  delete m;
  scn::timeline_dump();
}

// Builds ahead, on a worker thread and the Metadata's build stream, the rulebooks / plans the caller
// is about to request (ops: n_ops x 13 longs = kind, a[3], b[3], filter[3], stride[3]; kind 1 =
// submanifold(a = size), 2 = convolution(a = in, b = out), 3 = deconvolution(a = in (coarse),
// b = out (fine))).  Purely a hint: results are identical with or without it, entries are built
// in the same lazily-filled caches (Metadata.cpp:429-510) under the same keys; a failing hint is
// ignored and the error resurfaces when the caller requests that entry itself.
static void prefetch_worker(scn_metadata *m, int which) {
  struct Done { scn_metadata *m; int which; ~Done() { if (which == 0) m->md.set_chain_done(true); else { m->md.worker2Done.store(true); m->md.cv.notify_all(); } } } done{m, which};
  for (const PrefetchOp &op : (which == 0 ? m->ops : m->ops2)) {
    if (m->stop) break;
    const long *a = op.v + 1, *b = op.v + 4, *f = op.v + 7, *s = op.v + 10;
    struct Mark { const PrefetchOp &o; ~Mark() { scn::timeline_mark("worker", (int)o.v[0], o.v[1], o.v[7]); } } mark{op};
    if (op.v[0] == 0) {
      if (m->md.input_layer(m->inSz, m->inCoords, m->inOnDevice, m->inRows, m->inCols, m->inBatch, m->inMode)) break;
    } else if (op.v[0] == 1) {
      scn::SubmEntry *e;
      if (m->md.get_submanifold(a, f, &e)) break;
    } else if (op.v[0] == 2) {
      scn::ConvEntry *e;
      if (m->md.get_conv(a, b, f, s, &e)) break;
    } else if (op.v[0] == 3) {
      scn::ConvEntry *e = which == 1 ? m->md.wait_conv(b, f, s) : nullptr; // built by the chain worker
      if (m->stop) break;
      if (!e && m->md.get_conv(b, a, f, s, &e)) break;
      scn::Grid *gf = m->md.find_grid(b);
      if (scn::g_math_mode != 0 && scn::tc_available() && gf && gf->n > 0 && e->geom.M == 1 && e->rb.total == gf->n)
        if (m->md.get_deconv_plan(*e)) break;
    }
  }
}
// Two process-wide worker threads (chain / everything else) serve the prefetch jobs of all Metadata objects: a thread per
// forward cost ~0.2 ms before its first kernel (creation + binding the CUDA context), on the critical path of the forward.
namespace {
struct WorkerPool {
  std::mutex mu;
  std::condition_variable cv;
  std::deque<scn_metadata *> q[3];
};
WorkerPool *g_pool = nullptr; // never destroyed: the threads sleep on it until the process ends
std::once_flag g_pool_once;
void pool_main(int which) {
  scn::set_prefetch_worker_thread(true, which == 2 ? 0 : which); // thread 2 serves whole-Metadata jobs (reference grids) on their context 0
  int dev = -1;
  for (;;) {
    scn_metadata *m;
    {
      std::unique_lock<std::mutex> lk(g_pool->mu);
      g_pool->cv.wait(lk, [&] { return !g_pool->q[which].empty(); });
      m = g_pool->q[which].front();
      g_pool->q[which].pop_front();
    }
    if (dev != m->device) { cudaSetDevice(m->device); dev = m->device; }
    prefetch_worker(m, which == 2 ? 0 : which);
    { std::lock_guard<std::mutex> lk(m->jobMu); m->pending--; }
    m->jobCv.notify_all();
  }
}
void pool_submit(scn_metadata *m, int which) {
  std::call_once(g_pool_once, [] {
    g_pool = new WorkerPool();
    for (int w = 0; w < 3; w++) std::thread(pool_main, w).detach();
  });
  { std::lock_guard<std::mutex> lk(m->jobMu); m->pending++; }
  { std::lock_guard<std::mutex> lk(g_pool->mu); g_pool->q[which].push_back(m); }
  g_pool->cv.notify_all();
}
} // namespace
int scn_metadata_prefetch(scn_metadata *m, int n_ops, const long *ops) {
  if (!m) { scn::set_error("null scn_metadata handle"); return -3; }
  m->md.set_chain_done(true);
  wait_jobs(m);
  m->ops.clear();
  m->ops2.clear();
  // The strided convolutions create the grids level by level: that chain is the critical path, so it
  // gets a worker (and a build stream) of its own; submanifold plans and deconvolution plans only
  // hang off it and are built by a second worker on the second build context.
  // A strided convolution is on the chain when something hangs off its OUTPUT grid; the z-collapsing
  // convolutions at the end of the FPN are leaves and go to the second worker as well.
  auto key3 = [](const long *v) { return (v[0] << 42) ^ (v[1] << 21) ^ v[2]; };
  std::vector<long> usedAsInput;
  for (int i = 0; i < n_ops; i++) usedAsInput.push_back(key3(ops + i * 13 + (ops[i * 13] == 3 ? 4 : 1)));
  for (int i = 0; i < n_ops; i++) {
    PrefetchOp op;
    for (int j = 0; j < 13; j++) op.v[j] = ops[i * 13 + j];
    bool chain = op.v[0] == 2 && std::find(usedAsInput.begin(), usedAsInput.end(), key3(op.v + 4)) != usedAsInput.end();
    (m->md.nCtx >= 2 && !chain ? m->ops2 : m->ops).push_back(op);
  }
  // Second worker: shallow levels first.  Its entries become buildable as the chain worker descends
  // (a submanifold plan needs its grid, a deconvolution plan the convolution that created the coarse
  // grid); taken in request order it would sit on the deepest level's deconvolution plans while the
  // shallow ones -- buildable long before -- queue behind them.
  // Submanifold plans first (the bottom-up pass needs them level by level, as the chain worker descends), then what the
  // top-down pass and the z-collapsing convolutions need, deepest level first -- the order in which the network uses them.
  static const bool interleave = !(getenv("SCN_DECONV_EARLY") && atoi(getenv("SCN_DECONV_EARLY")) == 0);
  if (interleave) {
    // A deconvolution plan (coarse -> fine) becomes buildable together with the submanifold plans of its COARSE grid (the chain
    // worker has built the convolution fine -> coarse by then): it is built right behind them, while this worker would
    // otherwise idle until the next level's grid exists.  Taken after ALL submanifold plans (deepest first), the plans of
    // the large levels were finished last and the top-down pass waited for them (two ~50 us stalls on the caller's stream).
    std::stable_sort(m->ops2.begin(), m->ops2.end(), [](const PrefetchOp &x, const PrefetchOp &y) {
      auto cls = [](const PrefetchOp &o) { return o.v[0] == 2 ? 1 : 0; };               // leaf convolutions (z-collapse) last
      auto level = [](const PrefetchOp &o) { return o.v[1]; };                             // subm: its grid; deconv: its coarse grid; conv: its input grid
      if (cls(x) != cls(y)) return cls(x) < cls(y);
      if (cls(x) == 1) return level(x) < level(y);
      if (level(x) != level(y)) return level(x) > level(y);
      return (x.v[0] == 1) && (y.v[0] != 1);
    });
  } else
  std::stable_sort(m->ops2.begin(), m->ops2.end(), [](const PrefetchOp &x, const PrefetchOp &y) {
    auto fine = [](const PrefetchOp &o) { return o.v[0] == 3 ? o.v[4] : o.v[1]; }; // spatial size[0] of the (fine) grid the entry hangs off
    const bool sx = x.v[0] == 1, sy = y.v[0] == 1;
    if (sx != sy) return sx;
    return sx ? fine(x) > fine(y) : fine(x) < fine(y);
  });
  {
    std::lock_guard<std::mutex> lk(m->md.mapMu);
    for (const PrefetchOp &o : m->ops2)
      if (o.v[0] == 1) m->md.subm[scn::SubmKey{scn::P3{o.v[1], o.v[2], o.v[3]}, scn::P3{o.v[7], o.v[8], o.v[9]}}].assigned = true;
  }
  m->stop = false;
  m->md.set_chain_done(false);
  pool_submit(m, 0);
  if (!m->ops2.empty()) { m->md.worker2Done.store(false); pool_submit(m, 1); }
  return 0;
}

// Reference-numbered grids beside an internally numbered forward (program.cu): input layer + the given strided convolutions
// (ops: n_ops x 13 longs, kind 2), all on a worker thread; scn_metadata_wait_jobs blocks until they are built.
int scn_metadata_build_reference_grids(scn_metadata *m, const long sz[3], const long *coords, int on_device, long nrows, int ncols, int batch_size,
                                       int mode, int n_ops, const long *ops, void *coords_ready_event) {
  M_OR_FAIL(m);
  m->md.set_chain_done(true);
  wait_jobs(m);
  for (int d = 0; d < 3; d++) m->inSz[d] = sz[d];
  m->inCoords = coords; m->inOnDevice = on_device; m->inRows = nrows; m->inCols = ncols; m->inBatch = batch_size; m->inMode = mode;
  m->md.coordsReady = static_cast<cudaEvent_t>(coords_ready_event);
  // (stream priorities do not help: normal-priority streams for this job measured 5.39 vs 5.27 ms in round 1; in round 2 the layers on
  // a high-priority stream of their own with this job on lowest-priority streams: 5.19 vs 5.05 ms)
  m->ops.clear();
  m->ops2.clear();
  PrefetchOp in;
  for (int j = 0; j < 13; j++) in.v[j] = 0;
  m->ops.push_back(in);
  for (int i = 0; i < n_ops; i++) {
    PrefetchOp op;
    for (int j = 0; j < 13; j++) op.v[j] = ops[i * 13 + j];
    if (op.v[0] == 2) m->ops.push_back(op);
  }
  m->stop = false;
  m->md.set_chain_done(false);
  pool_submit(m, 2);
  return 0;
}
int scn_metadata_wait_jobs(scn_metadata *m) {
  M_OR_FAIL(m);
  wait_jobs(m);
  return 0;
}
int scn_input_layer_build(scn_metadata *m, const long sz[3], const long *coords, int on_device, long nrows, int ncols,
                          int batch_size, int mode, long *n_active, int *max_active) {
  M_OR_FAIL(m);
  scn::timeline_mark("input", 0, nrows, 0);
  SCN_TRY(m->md.input_layer(sz, coords, on_device, nrows, ncols, batch_size, mode));
  scn::timeline_mark("input", 1, nrows, 0);
  if (n_active) *n_active = m->md.input.nOut;
  if (max_active) *max_active = m->md.input.maxActive;
  return 0;
}
int scn_input_layer_built(scn_metadata *m, long *n_active, int *max_active) {
  if (!m || !m->md.input.valid) return 0;
  if (n_active) *n_active = m->md.input.nOut;
  if (max_active) *max_active = m->md.input.maxActive;
  return 1;
}
int scn_input_layer_forward(scn_metadata *m, const float *in, float *out, int C) {
  M_OR_FAIL(m);
  auto &I = m->md.input;
  SCN_CHECK(I.valid, "input layer not built");
  SCN_TRY(m->md.wait_ready(I.rdy));
  if (I.mode == 0) {
    SCN_CUDA(cudaMemcpyAsync(out, in, (size_t)I.nOut * C * 4, cudaMemcpyDeviceToDevice, m->md.cstream));
    return 0;
  }
  return scn::input_forward(in, out, I.nOut, I.maxActive, C, I.tab, I.mode == 4, m->md.cstream);
}
// InputLayer forward that also writes the rows as bfloat16 zero-padded to `padded` (16 or 32) channels: what the first
// convolution of a bf16-mode program gathers (modes 1-4; used by the program executor).
int scn_input_layer_forward_padded_bf16(scn_metadata *m, const float *in, float *out, void *out_bf16, int C, int padded) {
  M_OR_FAIL(m);
  auto &I = m->md.input;
  SCN_CHECK(I.valid && I.mode != 0 && padded >= C, "input layer not built / unsupported mode");
  SCN_TRY(m->md.wait_ready(I.rdy));
  return scn::input_forward_pad16(in, out, out_bf16, I.nOut, I.maxActive, C, padded, I.tab, I.mode == 4, m->md.cstream);
}
int scn_input_layer_backward(scn_metadata *m, float *din, const float *dout, int C) {
  M_OR_FAIL(m);
  auto &I = m->md.input;
  SCN_CHECK(I.valid, "input layer not built");
  SCN_TRY(m->md.wait_ready(I.rdy));
  if (I.mode == 0) {
    SCN_CUDA(cudaMemcpyAsync(din, dout, (size_t)I.nOut * C * 4, cudaMemcpyDeviceToDevice, m->md.cstream));
    return 0;
  }
  return scn::input_backward(din, dout, I.nIn, I.nOut, I.maxActive, C, I.tab, I.mode == 4, m->md.cstream);
}

// OutputLayer (CPU/IOLayers.cpp:97-140): the InputLayer's rule table run backwards WITHOUT averaging -- every input row receives
// the feature row of its voxel; its gradient sums the rows of a voxel.
int scn_output_layer_forward(scn_metadata *m, const float *in, float *out, int C) {
  M_OR_FAIL(m);
  auto &I = m->md.input;
  SCN_CHECK(I.valid, "input layer not built");
  SCN_TRY(m->md.wait_ready(I.rdy));
  if (I.mode == 0) {
    SCN_CUDA(cudaMemcpyAsync(out, in, (size_t)I.nOut * C * 4, cudaMemcpyDeviceToDevice, m->md.cstream));
    return 0;
  }
  return scn::input_backward(out, in, I.nIn, I.nOut, I.maxActive, C, I.tab, /*average=*/0, m->md.cstream);
}
int scn_output_layer_backward(scn_metadata *m, float *d_in, const float *d_out, int C) {
  M_OR_FAIL(m);
  auto &I = m->md.input;
  SCN_CHECK(I.valid, "input layer not built");
  SCN_TRY(m->md.wait_ready(I.rdy));
  if (I.mode == 0) {
    SCN_CUDA(cudaMemcpyAsync(d_in, d_out, (size_t)I.nOut * C * 4, cudaMemcpyDeviceToDevice, m->md.cstream));
    return 0;
  }
  return scn::input_forward(d_out, d_in, I.nOut, I.maxActive, C, I.tab, /*average=*/0, m->md.cstream);
}

// ---- internal row numbering (program replay): see Metadata::spatialIds
int scn_metadata_set_internal_numbering(scn_metadata *m, int on) {
  M_OR_FAIL(m);
  SCN_CHECK(!m->md.input.valid, "set the numbering before the input layer is built");
  m->md.spatialIds = on != 0;
  return 0;
}
namespace {
__global__ void k_row_permutation(const int4 *refCoords, int n, scn::GridView g, const int *p2id, int *perm) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int4 c = refCoords[i];
    const int p = scn::grid_lookup(g, c.x, c.y, c.z, c.w);
    perm[i] = p >= 0 ? p2id[p] : -1;
  }
}
__global__ void k_gather_rows(const float4 *__restrict__ src, float4 *__restrict__ dst, const int *__restrict__ perm, long rows, int c4) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < rows * c4; i += (long)gridDim.x * blockDim.x) {
    const long r = i / c4;
    const int s = perm[r];
    dst[i] = s >= 0 ? src[(long)s * c4 + (i - r * c4)] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
} // namespace
// dst[id] = src[row of the same site in `internal`] for the grid of spatial size sz: rows of a feature matrix computed in the
// internal numbering of `internal` are handed out in the reference numbering of `ref` (both built from the same input).
// Runs on ref's compute stream; cols % 4 == 0.
int scn_rows_to_reference_order(scn_metadata *ref, scn_metadata *internal, const long sz[3], const float *src, float *dst, int cols) {
  M_OR_FAIL(ref);
  M_OR_FAIL(internal);
  scn::Grid *gr = ref->md.find_grid(sz), *gi = internal->md.find_grid(sz);
  SCN_CHECK(gr && gi && gr->n == gi->n && cols % 4 == 0, "rows_to_reference_order: grids differ");
  if (gr->n == 0) return 0;
  cudaStream_t s = ref->md.cstream;
  SCN_TRY(ref->md.wait_ready(gr->rdy));
  if (gi->rdy.ev) SCN_CUDA(cudaStreamWaitEvent(s, gi->rdy.ev, 0));
  int *perm = nullptr;
  SCN_CUDA(cudaMallocAsync((void **)&perm, (size_t)gr->n * 4, s));
  const scn::GridView v{gi->dir, gi->bmask, gi->wbase, gi->dd[0], gi->dd[1], gi->dd[2], gi->dirCells, (int)gi->sz[0], (int)gi->sz[1], (int)gi->sz[2]};
  k_row_permutation<<<scn::stream_grid(gr->n, 256), 256, 0, scn::LS(s)>>>(gr->coords, gr->n, v, gi->p2id, perm);
  k_gather_rows<<<scn::stream_grid((long)gr->n * cols / 4, 256), 256, 0, scn::LS(s)>>>(reinterpret_cast<const float4 *>(src), reinterpret_cast<float4 *>(dst), perm,
                                                                                       gr->n, cols / 4);
  SCN_CUDA(cudaGetLastError());
  cudaFreeAsync(perm, s);
  return 0;
}
// The same for SEVERAL feature matrices in ONE launch (the end of a replayed forward hands out 5 small maps: five pairs of
// launches, five stream-ordered allocations and the host time between them were 0.2 ms of a 4.9 ms forward).  One warp per
// destination row: lane 0 looks the row's site up in the internal grid, the warp copies the row.
namespace {
constexpr int kMaxOutMaps = 8;
struct OutMap { const int4 *refCoords; const int *p2id; const float4 *src; float4 *dst; scn::GridView g; int n, c4, firstWarp; };
struct OutMaps { OutMap m[kMaxOutMaps]; int count, totalWarps, scatter; }; // scatter: dst[internal row] = src[reference row] (gradients on their way in)
__global__ void __launch_bounds__(256) k_rows_to_reference_multi(OutMaps P) {
  scn::pdl_launch_dependents();
  scn::pdl_wait();
  const int lane = threadIdx.x & 31;
  for (int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < P.totalWarps; w += gridDim.x * (blockDim.x >> 5)) {
    int k = 0;
    while (k + 1 < P.count && w >= P.m[k + 1].firstWarp) k++;
    const OutMap &M = P.m[k];
    const int row = w - M.firstWarp;
    int srcRow = -1;
    if (lane == 0) {
      const int4 c = M.refCoords[row];
      const int p = scn::grid_lookup(M.g, c.x, c.y, c.z, c.w);
      srcRow = p >= 0 ? M.p2id[p] : -1;
    }
    srcRow = __shfl_sync(0xffffffffu, srcRow, 0);
    if (P.scatter) {
      if (srcRow >= 0) for (int j = lane; j < M.c4; j += 32) M.dst[(long)srcRow * M.c4 + j] = M.src[(long)row * M.c4 + j];
      continue;
    }
    for (int j = lane; j < M.c4; j += 32) M.dst[(long)row * M.c4 + j] = srcRow >= 0 ? M.src[(long)srcRow * M.c4 + j] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
static int rows_reorder_multi(scn_metadata *ref, scn_metadata *internal, int n_maps, const long *sizes, const float *const *src, float *const *dst,
                              const int *cols, int scatter);
} // namespace
int scn_rows_to_reference_order_multi(scn_metadata *ref, scn_metadata *internal, int n_maps, const long *sizes, const float *const *src, float *const *dst,
                                      const int *cols) {
  return rows_reorder_multi(ref, internal, n_maps, sizes, src, dst, cols, 0);
}
int scn_rows_from_reference_order(scn_metadata *ref, scn_metadata *internal, const long size[3], const float *src, float *dst, int cols) {
  return rows_reorder_multi(ref, internal, 1, size, &src, &dst, &cols, 1);
}
namespace {
static int rows_reorder_multi(scn_metadata *ref, scn_metadata *internal, int n_maps, const long *sizes, const float *const *src, float *const *dst,
                              const int *cols, int scatter) {
  M_OR_FAIL(ref);
  M_OR_FAIL(internal);
  SCN_CHECK(n_maps >= 0 && n_maps <= kMaxOutMaps, "rows_to_reference_order_multi: at most 8 maps per call");
  OutMaps P;
  P.count = 0;
  P.totalWarps = 0;
  cudaStream_t s = ref->md.cstream;
  for (int i = 0; i < n_maps; i++) {
    scn::Grid *gr = ref->md.find_grid(sizes + 3 * i), *gi = internal->md.find_grid(sizes + 3 * i);
    SCN_CHECK(gr && gi && gr->n == gi->n && cols[i] % 4 == 0, "rows_to_reference_order: grids differ");
    if (gr->n == 0) continue;
    SCN_TRY(ref->md.wait_ready(gr->rdy));
    if (gi->rdy.ev) SCN_CUDA(cudaStreamWaitEvent(s, gi->rdy.ev, 0));
    OutMap &M = P.m[P.count++];
    M.refCoords = gr->coords;
    M.p2id = gi->p2id;
    M.src = reinterpret_cast<const float4 *>(src[i]);
    M.dst = reinterpret_cast<float4 *>(dst[i]);
    M.g = scn::GridView{gi->dir, gi->bmask, gi->wbase, gi->dd[0], gi->dd[1], gi->dd[2], gi->dirCells, (int)gi->sz[0], (int)gi->sz[1], (int)gi->sz[2]};
    M.n = gr->n;
    M.c4 = cols[i] / 4;
    M.firstWarp = P.totalWarps;
    P.totalWarps += gr->n;
  }
  if (P.totalWarps == 0) return 0;
  P.scatter = scatter;
  SCN_CUDA(scn::launch_pdl(k_rows_to_reference_multi, dim3(std::min(scn::cdiv(P.totalWarps, 8), 148 * 8)), dim3(256), 0, scn::LS(s), P));
  SCN_CUDA(cudaGetLastError());
  return 0;
}
} // namespace
int scn_get_batch_size(scn_metadata *m, const long sz[3], int *batch) {
  M_OR_FAIL(m);
  scn::Grid *g = m->md.find_grid(sz);
  *batch = g ? g->batch : 0;
  return 0;
}
int scn_get_nactive(scn_metadata *m, const long sz[3], long *n) {
  M_OR_FAIL(m);
  scn::Grid *g = m->md.find_grid(sz);
  *n = g ? g->n : 0; // Metadata::getNActive default-constructs 0 for unknown sizes
  return 0;
}
int scn_get_spatial_locations(scn_metadata *m, const long sz[3], long *out, int on_device) {
  M_OR_FAIL(m);
  return m->md.spatial_locations(sz, out, on_device);
}
int scn_submanifold_prepare(scn_metadata *m, const long sz[3], const long f[3], long *n_rules) {
  M_OR_FAIL(m);
  scn::SubmEntry *e;
  SCN_TRY(m->md.get_submanifold(sz, f, &e));
  if (n_rules) *n_rules = e->rb.total;
  return 0;
}
int scn_convolution_prepare(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long s[3], long *n_out,
                            long *n_rules) {
  M_OR_FAIL(m);
  scn::ConvEntry *e;
  SCN_TRY(m->md.get_conv(inS, outS, f, s, &e));
  SCN_CHECK(e->out == (scn::P3{outS[0], outS[1], outS[2]}), "this (input size, filter, stride) rulebook was built for another output size");
  if (n_out) *n_out = m->md.find_grid(outS)->n;
  if (n_rules) *n_rules = e->rb.total;
  return 0;
}

// getSparseToDenseRuleBook (Metadata.cpp:469-483; ConvolutionRules.h:109-151): per batch item the pairs (row, spatial offset) of its
// sites in hash-iteration order, offset = RectangularRegion::offset over the whole spatial size (last dimension fastest).
__global__ void k_s2d_rules(const int *__restrict__ rank2id, const int4 *__restrict__ coords, int n, int sy, int sz, int2 *__restrict__ pairs) {
  for (long r = blockIdx.x * (long)blockDim.x + threadIdx.x; r < n; r += (long)gridDim.x * blockDim.x) {
    const int id = rank2id[r];
    const int4 c = coords[id];
    pairs[r] = make_int2(id, (c.x * sy + c.y) * sz + c.z);
  }
}
static int s2d_rulebook(scn_metadata *m, const long a[3], scn::RuleBookDev **out) {
  const scn::P3 key{a[0], a[1], a[2]};
  auto it = m->s2d.find(key);
  if (it != m->s2d.end()) { *out = &it->second; return 0; }
  scn::Grid *g = m->md.find_grid(a);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  SCN_CHECK(a[0] * a[1] * a[2] < (1l << 31), "spatial volume exceeds the int32 rule format");
  scn::Metadata::BuildLock bl(m->md);
  SCN_TRY(m->md.ensure_rank(*g));
  scn::RuleBookDev rb;
  rb.nLists = g->batch;
  rb.total = g->n;
  rb.off.assign(1, 0);
  for (int b = 0; b < g->batch; b++) rb.off.push_back(rb.off.back() + g->itemCount[b]);
  rb.pairs = m->md.alloc_n<int2>(std::max(1, g->n));
  SCN_CHECK(rb.pairs, "alloc");
  cudaStream_t s = m->md.cur().stream;
  if (g->n) k_s2d_rules<<<scn::stream_grid(g->n, 256), 256, 0, scn::LS(s)>>>(g->rank2id, g->coords, g->n, (int)a[1], (int)a[2], rb.pairs);
  SCN_CUDA(cudaStreamSynchronize(s));
  *out = &(m->s2d[key] = rb);
  return 0;
}
static int find_rb(scn_metadata *m, int kind, const long a[3], const long b[3], const long c[3], scn::RuleBookDev **rb) {
  if (kind == 3) return s2d_rulebook(m, a, rb);
  if (kind == 1) {
    scn::SubmEntry *e = nullptr;
    {
      std::lock_guard<std::mutex> lk(m->md.mapMu);
      auto it = m->md.subm.find(scn::SubmKey{scn::P3{a[0], a[1], a[2]}, scn::P3{b[0], b[1], b[2]}});
      SCN_CHECK(it != m->md.subm.end() && it->second.rdy.ready, "submanifold rulebook not built");
      e = &it->second;
    }
    SCN_TRY(m->md.ensure_subm_rules(*e));
    *rb = &e->rb;
    return 0;
  }
  scn::ConvEntry *ce = nullptr;
  {
    std::lock_guard<std::mutex> lk(m->md.mapMu);
    auto it = m->md.conv.find(scn::ConvKey{scn::P3{a[0], a[1], a[2]}, scn::P3{b[0], b[1], b[2]}, scn::P3{c[0], c[1], c[2]}});
    SCN_CHECK(it != m->md.conv.end() && it->second.rdy.ready, "convolution rulebook not built");
    ce = &it->second;
  }
  SCN_TRY(m->md.ensure_conv_rules(*ce));
  *rb = &ce->rb;
  return 0;
}
int scn_rulebook_info(scn_metadata *m, int kind, const long a[3], const long b[3], const long c[3], int *n_lists, long *list_len) {
  M_OR_FAIL(m);
  if (kind == 0) {
    auto &I = m->md.input;
    SCN_CHECK(I.valid, "input layer not built");
    *n_lists = I.mode == 0 ? 1 : 2;
    if (list_len) { list_len[0] = 4; if (I.mode) list_len[1] = (long)I.nOut * (1 + I.maxActive); }
    return 0;
  }
  scn::RuleBookDev *rb;
  SCN_TRY(find_rb(m, kind, a, b, c, &rb));
  *n_lists = rb->nLists;
  if (list_len) for (int i = 0; i < rb->nLists; i++) list_len[i] = 2l * (rb->off[i + 1] - rb->off[i]);
  return 0;
}
int scn_rulebook_copy(scn_metadata *m, int kind, const long a[3], const long b[3], const long c[3], int list, int *dst) {
  M_OR_FAIL(m);
  cudaStream_t s = m->md.cur().stream;
  if (kind == 0) {
    auto &I = m->md.input;
    SCN_CHECK(I.valid, "input layer not built");
    if (list == 0) { dst[0] = I.mode; dst[1] = I.maxActive; dst[2] = I.nIn; dst[3] = I.nOut; return 0; }
    SCN_CHECK(I.mode != 0 && list == 1, "list index");
    SCN_CUDA(cudaMemcpyAsync(dst, I.tab, (size_t)I.nOut * (1 + I.maxActive) * 4, cudaMemcpyDeviceToHost, s));
    SCN_CUDA(cudaStreamSynchronize(s));
    return 0;
  }
  scn::RuleBookDev *rb;
  SCN_TRY(find_rb(m, kind, a, b, c, &rb));
  SCN_CHECK(list >= 0 && list < rb->nLists, "list index");
  long n = rb->off[list + 1] - rb->off[list];
  if (n) {
    SCN_CUDA(cudaMemcpyAsync(dst, rb->pairs + rb->off[list], n * 8, cudaMemcpyDeviceToHost, s));
    SCN_CUDA(cudaStreamSynchronize(s));
  }
  return 0;
}
int scn_iteration_order(scn_metadata *m, const long sz[3], int *dst) {
  M_OR_FAIL(m);
  scn::Grid *g = m->md.find_grid(sz);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  scn::Metadata::BuildLock bl(m->md);
  SCN_TRY(m->md.ensure_rank(*g));
  if (g->n) {
    SCN_CUDA(cudaMemcpyAsync(dst, g->rank2id, (size_t)g->n * 4, cudaMemcpyDeviceToHost, m->md.cur().stream));
    SCN_CUDA(cudaStreamSynchronize(m->md.cur().stream));
  }
  return 0;
}

static bool tc_ok(int Cin, int Cout, int K) {
  return scn::g_math_mode != 0 && scn::tc_available() && Cout % 32 == 0 && Cout >= 32 && Cout <= 256 && K <= 64 && Cin >= 4 && Cin <= 1024;
}
// out += addend (optional) and the bf16 copy of out (optional), for the paths whose kernels do not fuse them
static int plain_epilogue(float *out, const float *addend, void *out16, long rows, int C, cudaStream_t s) {
  if (rows <= 0) return 0;
  if (addend) return scn::add_rows(out, addend, out, rows * C, s, out16);
  if (out16) return scn::to_bf16(out, out16, rows * C, s);
  return 0;
}
static int run_plan(Metadata &M, const scn::NbrPlan &plan, const float *in, float *out, const float *w, const float *bias, int Cin, int Cout,
                    long nInRows, const void *in16, long long wTag, const float *addend, void *out16) {
  if (tc_ok(Cin, Cout, plan.K))
    return scn::launch_conv_plan_tc(in, out, w, plan.nbr, plan.outRow, plan.tileMask, plan.nOut, plan.K, Cin, Cout, bias, scn::g_math_mode, M.cstream,
                                    nullptr, plan.K, nInRows, in16, wTag, addend, out16, plan.nOut);
  SCN_CHECK(in && out, "CUDA-core path needs the fp32 rows");
  SCN_TRY(scn::launch_conv_plan_simt(in, out, w, plan.nbr, plan.outRow, plan.nOut, plan.K, Cin, Cout, bias, M.cstream));
  return plain_epilogue(out, addend, out16, plan.nOut, Cout, M.cstream);
}

int scn_submanifold_convolution_forward(scn_metadata *m, const long sz[3], const long f[3], const float *in, float *out, const float *w,
                                        const float *bias, int Cin, int Cout, double *macs, const void *in_bf16, long long weight_tag,
                                        const float *add_in, void *out_bf16) {
  M_OR_FAIL(m);
  scn::SubmEntry *e;
  SCN_TRY(m->md.get_submanifold(sz, f, &e));
  if (macs) *macs = (double)e->rb.total * Cin * Cout;
  SCN_TRY(m->md.wait_ready(e->rdy));
  return run_plan(m->md, e->plan, in, out, w, bias, Cin, Cout, m->md.find_grid(sz)->n, in_bf16, weight_tag, add_in, out_bf16);
}
int scn_convolution_forward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in,
                            float *out, const float *w, const float *bias, int Cin, int Cout, double *macs, const void *in_bf16, long long weight_tag,
                              const float *add_in, void *out_bf16) {
  M_OR_FAIL(m);
  scn::ConvEntry *e;
  SCN_TRY(m->md.get_conv(inS, outS, f, st, &e));
  if (macs) *macs = (double)e->rb.total * Cin * Cout;
  SCN_TRY(m->md.wait_ready(e->rdy));
  return run_plan(m->md, e->plan, in, out, w, bias, Cin, Cout, m->md.find_grid(inS)->n, in_bf16, weight_tag, add_in, out_bf16);
}
__global__ void k_fill_rows_bias(float *out, long n, int C, const float *bias) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n * C; i += (long)gridDim.x * blockDim.x) out[i] = bias ? bias[i % C] : 0.f;
}
int scn_deconvolution_forward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in,
                              float *out, const float *w, const float *bias, int Cin, int Cout, double *macs, const void *in_bf16, long long weight_tag,
                              const float *add_in, void *out_bf16) {
  M_OR_FAIL(m);
  // CPU/Deconvolution.cpp:15-16: the rulebook of the convolution outS -> inS
  scn::ConvEntry *e;
  SCN_TRY(m->md.get_conv(outS, inS, f, st, &e));
  if (macs) *macs = (double)e->rb.total * Cin * Cout;
  scn::Grid *gf = m->md.find_grid(outS);
  SCN_CHECK(gf, "output grid");
  cudaStream_t s = m->md.cstream;
  // every fine row with a parent is written exactly once when each input site has one output cell
  bool single = e->rb.total == gf->n && !bias;
  if (single && e->geom.M == 1 && tc_ok(Cin, Cout, 1) && gf->n > 0) {
    SCN_TRY(m->md.get_deconv_plan(*e));
    SCN_TRY(m->md.wait_ready(e->deconvRdy));
    const scn::DeconvPlan &d = e->deconv;
    return scn::launch_conv_plan_tc(in, out, w, d.nbr, d.outRow, d.tileMask, d.nTiles * 128, 1, Cin, Cout, nullptr, scn::g_math_mode, s, d.tileW,
                                    e->rb.nLists, m->md.find_grid(inS)->n, in_bf16, weight_tag, add_in, out_bf16, gf->n);
  }
  SCN_CHECK(in && out, "CUDA-core deconvolution needs the fp32 rows");
  SCN_TRY(m->md.ensure_conv_rules(*e));
  SCN_TRY(m->md.wait_ready(e->rdy));
  SCN_TRY(m->md.wait_ready(e->rulesRdy));
  if (!single && gf->n) k_fill_rows_bias<<<scn::stream_grid((long)gf->n * Cout, 256), 256, 0, scn::LS(s)>>>(out, gf->n, Cout, bias);
  SCN_TRY(scn::launch_conv_list_simt(in, out, w, e->rb.pairs, e->rb.d_off, e->rb.off.data(), e->rb.nLists, Cin, Cout, /*srcIsY=*/1, single ? 1 : 0, s));
  return plain_epilogue(out, add_in, out_bf16, gf->n, Cout, s);
}

// d_in = forward tensor-core convolution of d_out with transposed weights (conv_bwd.cu header).  W: [K][Cin][Cout] of the
// FORWARD layer; d_out rows have Cout channels (nSrcRows of them), d_in rows Cin channels (nDstRows, all written by the plan).
static int dIn_tensor_core(Metadata &M, const float *d_out, float *d_in, const float *W, int K, int Cin, int Cout, int reverse, const int *nbr,
                           const int *outRow, const unsigned long long *tileMask, int nOutPlan, const int *tileW, long nSrcRows, long nDstRows,
                           const void *dout16 = nullptr) {
  cudaStream_t s = M.cstream;
  // the transposed (and, for the symmetric submanifold plan, offset-reversed) weights are read in place by the operand-image kernel
  return scn::launch_conv_plan_tc(d_out, d_in, W, nbr, outRow, tileMask, nOutPlan, tileW ? 1 : K, /*Cin=*/Cout, /*Cout=*/Cin, nullptr, scn::g_math_mode, s, tileW, K,
                                  nSrcRows, dout16, 0, nullptr, nullptr, nDstRows, 0, reverse ? 2 : 1);
}
// bf16 mode: one bf16 copy of d_out serves both gradient kernels of a backward call (each used to make its own)
static int shared_dout16(cudaStream_t s, const float *d_out, long rows, int Cin, int Cout, const void **out) {
  *out = nullptr;
  if (scn::g_math_mode != 2 || !scn::tc_available() || rows == 0 || Cout % 32 != 0 || !tc_ok(Cout, Cin, 1)) return 0;
  return scn::dout_bf16_copy(d_out, rows * Cout, s, out);
}
int scn_submanifold_convolution_backward(scn_metadata *m, const long sz[3], const long f[3], const float *in, float *d_in, const float *d_out,
                                         const float *w, float *dw, float *d_bias, int Cin, int Cout) {
  const void *in16 = scn::bwd_in16_take(), *dout16 = nullptr;
  M_OR_FAIL(m);
  scn::SubmEntry *e;
  SCN_TRY(m->md.get_submanifold(sz, f, &e));
  scn::Grid *g = m->md.find_grid(sz);
  // d_in on the tensor cores: the plan of an odd filter is symmetric, d_in[q] = sum_j d_out[nbr[q][j]] @ W[K-1-j]^T
  const bool tcIn = d_in && tc_ok(Cout, Cin, e->plan.K) && f[0] % 2 == 1 && f[1] % 2 == 1 && f[2] % 2 == 1 && g->n > 0;
  // the per-offset rule lists (reference order) are only materialised when a CUDA-core kernel needs them: both tensor-core
  // gradient kernels read the execution plan
  const bool lists = !((tcIn || !d_in) && scn::dw_plan_ok(Cin, Cout, e->plan.K, scn::g_math_mode));
  if (lists) SCN_TRY(m->md.ensure_subm_rules(*e));
  SCN_TRY(m->md.wait_ready(e->rdy));
  if (lists) SCN_TRY(m->md.wait_ready(e->rulesRdy));
  SCN_TRY(shared_dout16(m->md.cstream, d_out, g->n, Cin, Cout, &dout16));
  if (tcIn) SCN_TRY(dIn_tensor_core(m->md, d_out, d_in, w, e->plan.K, Cin, Cout, /*reverse=*/1, e->plan.nbr, e->plan.outRow, e->plan.tileMask, e->plan.nOut, nullptr, g->n, g->n, dout16));
  return scn::conv_backward_simt(in, d_in, d_out, w, dw, d_bias, lists ? e->rb.pairs : nullptr, e->rb.d_off, lists ? e->rb.off.data() : nullptr, e->plan.K, g->n, g->n, Cin, Cout, 0, m->md.cstream, tcIn || !d_in, scn::g_math_mode, in16, dout16,
                                 e->plan.nbr, e->plan.outRow, e->plan.tileMask, e->plan.nOut); // d_in == NULL: input gradient not wanted
}
int scn_convolution_backward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in,
                             float *d_in, const float *d_out, const float *w, float *dw, float *d_bias, int Cin, int Cout) {
  const void *in16 = scn::bwd_in16_take(), *dout16 = nullptr;
  M_OR_FAIL(m);
  scn::ConvEntry *e;
  SCN_TRY(m->md.get_conv(inS, outS, f, st, &e));
  // d_in (fine rows) on the tensor cores: a deconvolution of d_out with W^T over the single-parent plan
  scn::Grid *gf = m->md.find_grid(inS), *gc = m->md.find_grid(outS);
  const bool tcIn = tc_ok(Cout, Cin, 1) && e->geom.M == 1 && e->rb.total == gf->n && gf->n > 0;
  const bool lists = !(tcIn && scn::dw_plan_ok(Cin, Cout, e->plan.K, scn::g_math_mode));
  if (lists) SCN_TRY(m->md.ensure_conv_rules(*e));
  SCN_TRY(m->md.wait_ready(e->rdy));
  if (lists) SCN_TRY(m->md.wait_ready(e->rulesRdy));
  SCN_TRY(shared_dout16(m->md.cstream, d_out, gc->n, Cin, Cout, &dout16));
  if (tcIn) {
    SCN_TRY(m->md.get_deconv_plan(*e));
    SCN_TRY(m->md.wait_ready(e->deconvRdy));
    const scn::DeconvPlan &d = e->deconv;
    SCN_TRY(dIn_tensor_core(m->md, d_out, d_in, w, e->rb.nLists, Cin, Cout, /*reverse=*/0, d.nbr, d.outRow, d.tileMask, d.nTiles * 128, d.tileW, gc->n, gf->n, dout16));
  }
  return scn::conv_backward_simt(in, d_in, d_out, w, dw, d_bias, lists ? e->rb.pairs : nullptr, e->rb.d_off, lists ? e->rb.off.data() : nullptr, e->plan.K, gf->n, gc->n, Cin, Cout, 0, m->md.cstream, tcIn, scn::g_math_mode, in16, dout16,
                                 e->plan.nbr, e->plan.outRow, e->plan.tileMask, e->plan.nOut);
}
int scn_deconvolution_backward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in,
                               float *d_in, const float *d_out, const float *w, float *dw, float *d_bias, int Cin, int Cout) {
  const void *in16 = scn::bwd_in16_take(), *dout16 = nullptr;
  M_OR_FAIL(m);
  scn::ConvEntry *e;
  SCN_TRY(m->md.get_conv(outS, inS, f, st, &e));
  // d_in (coarse rows) on the tensor cores: the strided convolution fine -> coarse of d_out with W^T
  scn::Grid *gc = m->md.find_grid(inS), *gf = m->md.find_grid(outS);
  const bool tcIn = tc_ok(Cout, Cin, e->plan.K) && gc->n > 0;
  const bool lists = !(tcIn && scn::dw_plan_ok(Cin, Cout, e->plan.K, scn::g_math_mode));
  if (lists) SCN_TRY(m->md.ensure_conv_rules(*e));
  SCN_TRY(m->md.wait_ready(e->rdy));
  if (lists) SCN_TRY(m->md.wait_ready(e->rulesRdy));
  SCN_TRY(shared_dout16(m->md.cstream, d_out, gf->n, Cin, Cout, &dout16));
  if (tcIn) SCN_TRY(dIn_tensor_core(m->md, d_out, d_in, w, e->plan.K, Cin, Cout, /*reverse=*/0, e->plan.nbr, e->plan.outRow, e->plan.tileMask, e->plan.nOut, nullptr, gf->n, gc->n, dout16));
  return scn::conv_backward_simt(in, d_in, d_out, w, dw, d_bias, lists ? e->rb.pairs : nullptr, e->rb.d_off, lists ? e->rb.off.data() : nullptr, e->plan.K, gc->n, gf->n, Cin, Cout, 1, m->md.cstream, tcIn, scn::g_math_mode, in16, dout16,
                                 e->plan.nbr, e->plan.outRow, e->plan.tileMask, e->plan.nOut);
}

// ---- NetworkInNetwork: a 1x1 "convolution" = dense GEMM over the feature rows, no Metadata involved
static int dense_rows_gemm(const float *in, float *out, const float *w, const float *bias, long n, int Cin, int Cout, cudaStream_t s, const void *in16, long long tag) {
  if (n == 0) return 0;
  SCN_CHECK(n < (1l << 31) - 256, "too many rows");
  if (tc_ok(Cin, Cout, 1)) // the tensor-core gather-GEMM with the identity plan (site p reads row p, writes row p)
    return scn::launch_conv_plan_tc(in, out, w, nullptr, nullptr, nullptr, (int)n, 1, Cin, Cout, bias, scn::g_math_mode, s, nullptr, 1, n, in16, tag, nullptr, nullptr, n);
  return scn::launch_conv_plan_simt(in, out, w, nullptr, nullptr, (int)n, 1, Cin, Cout, bias, s);
}
int scn_network_in_network_forward(const float *in, float *out, const float *weight, const float *bias, long n_rows, int n_in, int n_out, double *macs,
                                   void *stream, const void *in_bf16, long long weight_tag) {
  SCN_CHECK(n_rows >= 0 && n_in > 0 && n_out > 0 && (n_rows == 0 || (in && out && weight)), "NetworkInNetwork arguments");
  if (macs) *macs = (double)n_rows * n_in * n_out; // CPU/NetworkInNetwork.cpp:23
  return dense_rows_gemm(in, out, weight, bias, n_rows, n_in, n_out, static_cast<cudaStream_t>(stream), in_bf16, weight_tag);
}
int scn_network_in_network_backward_input(float *d_in, const float *d_out, const float *weight, long n_rows, int n_in, int n_out, void *stream) {
  SCN_CHECK(n_rows >= 0 && n_in > 0 && n_out > 0, "NetworkInNetwork arguments");
  if (n_rows == 0) return 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float *Wt = nullptr;
  SCN_CUDA(cudaMallocAsync((void **)&Wt, (size_t)n_in * n_out * 4, s));
  int r = scn::transpose_weights(weight, Wt, 1, n_in, n_out, 0, s);
  if (r == 0) r = dense_rows_gemm(d_out, d_in, Wt, nullptr, n_rows, n_out, n_in, s, nullptr, 0);
  cudaFreeAsync(Wt, s);
  return r;
}
int scn_network_in_network_backward_params(const float *in, const float *d_out, float *d_weight, float *d_bias, long n_rows, int n_in, int n_out, void *stream) {
  SCN_CHECK(n_rows >= 0 && n_in > 0 && n_out > 0 && d_weight, "NetworkInNetwork arguments");
  return scn::dense_rows_dw(in, d_out, d_weight, d_bias, n_rows, n_in, n_out, static_cast<cudaStream_t>(stream));
}

int scn_batchnorm_forward(const float *in, float *out, long n, int C, float *save_mean, float *save_invstd, float *running_mean,
                          float *running_var, const float *weight, const float *bias, float eps, float momentum, int mode, float leak,
                          void *stream, void *out_bf16) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SCN_CHECK(mode >= 0 && mode <= 2, "mode");
  // persistent, zero-initialised workspace per stream (calls on one stream are ordered; the
  // finalize kernel re-zeroes the statistics): no allocation, no memset per call
  static std::mutex mu;
  static std::vector<std::pair<std::pair<int, cudaStream_t>, void *>> cache; // keyed by (device, stream): stream handle 0 means "default" on every device
  constexpr int kMaxC = scn::kBnMaxC;
  SCN_CHECK(C <= kMaxC, "BatchNorm: too many channels");
  void *ws = nullptr;
  {
    int dev = 0;
    SCN_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    for (auto &e : cache) if (e.first.first == dev && e.first.second == s) ws = e.second;
    if (!ws) {
      SCN_CUDA(cudaMalloc(&ws, scn::kBnWorkspaceBytes));
      SCN_CUDA(cudaMemset(ws, 0, scn::kBnWorkspaceBytes));
      cache.emplace_back(std::make_pair(dev, s), ws);
    }
  }
  return scn::bn_forward(in, out, n, C, save_mean, save_invstd, running_mean, running_var, weight, bias, eps, momentum, mode, leak, ws, s, out_bf16);
}
extern "C++" {
namespace scn {
// (out may be NULL when out_bf16 is given: only the sign of the output is read)
int batchnorm_backward_y16(const float *in, float *d_in, const float *out, const void *out_bf16, float *d_out, long n, int C, const float *save_mean,
                           const float *save_invstd, const float *weight, float *d_weight, float *d_bias, float leak, cudaStream_t s) {
  void *ws = nullptr;
  SCN_CUDA(cudaMallocAsync(&ws, (size_t)C * 24 + 64, s));
  int r = bn_backward(in, d_in, out, d_out, n, C, save_mean, save_invstd, weight, d_weight, d_bias, leak, ws, s, out_bf16);
  cudaFreeAsync(ws, s);
  return r;
}
} // namespace scn
} // extern "C++"
int scn_batchnorm_backward(const float *in, float *d_in, const float *out, float *d_out, long n, int C, const float *save_mean,
                           const float *save_invstd, const float *weight, float *d_weight, float *d_bias, float leak, void *stream) {
  return scn::batchnorm_backward_y16(in, d_in, out, nullptr, d_out, n, C, save_mean, save_invstd, weight, d_weight, d_bias, leak, static_cast<cudaStream_t>(stream));
}
int scn_add_features(const float *a, const float *b, float *out, long n, void *stream, void *out_bf16) {
  return scn::add_rows(a, b, out, n, static_cast<cudaStream_t>(stream), out_bf16);
}
}
