// Metadata: GPU construction of active-site grids, the reference row numbering, the reference
// hash-iteration order (dense_hash_map emulation), rulebooks in the reference's format and the
// output-stationary execution plans.  See DESIGN.md "Rulebook build".
#include "metadata.cuh"
#include <stdlib.h>
#include <algorithm>
#include <limits.h>
#include <string.h>

namespace scn {

static thread_local std::string g_err;
void set_error(const std::string &m) { g_err = m; }
const char *last_error() { return g_err.c_str(); }

// ------------------------------------------------------------------ memory
// pinned scratch blocks are recycled across Metadata objects: cudaMallocHost costs milliseconds and a
// fresh Metadata is created for every forward (sparseconvnet/ioLayers.py:52-55)
static std::vector<int *> g_pinned_free;
static std::mutex g_pool_mu; // the recycling lists (pinned blocks, streams, events, chunks) are shared by all Metadata objects
static int *pinned_get() {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  if (!g_pinned_free.empty()) { int *p = g_pinned_free.back(); g_pinned_free.pop_back(); return p; }
  int *p = nullptr;
  if (cudaMallocHost(&p, 256 * 4) != cudaSuccess) return nullptr;
  return p;
}
// Device memory of a Metadata comes from a process-wide list of chunks that are never handed back to
// the driver.  The CUDA stream-ordered pool was measured to stall for 2-9 ms per call here: every
// Metadata allocates on its own build stream and is freed while the next one is already building on
// another stream, so the pool cannot reuse the blocks and maps fresh memory each forward.  A chunk
// carries the event that marks the end of its previous owner's work; the next owner's build stream
// waits for that event before the first use.
static std::vector<Chunk> g_chunks;
static size_t g_chunk_bytes = 0;       // idle chunks
static long g_chunk_mallocs = 0, g_chunk_waits = 0;
std::atomic<int> g_pool_growth{0};
void set_pool_growth(int on) { g_pool_growth.store(on); }
long debug_chunk_mallocs() { return g_chunk_mallocs; }
long debug_chunk_waits() { return g_chunk_waits; }
static size_t g_chunk_bytes_total = 0; // every chunk ever taken from the driver and not returned
constexpr size_t kChunkKeep = 32ull << 30; // beyond this much idle memory, chunks go back to the driver
long debug_chunk_total_mb() { return (long)(g_chunk_bytes_total >> 20); }
// hands every idle chunk back to the driver (the caller has synchronised the device) -> bytes released
long release_idle_chunks() {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  long freed = 0;
  for (Chunk &k : g_chunks) {
    if (k.freed) { cudaEventSynchronize(k.freed); cudaEventDestroy(k.freed); }
    cudaFree(k.p);
    freed += (long)k.cap;
    g_chunk_bytes_total -= k.cap;
  }
  g_chunks.clear();
  g_chunk_bytes = 0;
  return freed;
}
constexpr size_t kChunkGrow = 16ull << 30; // below this total, a new chunk is allocated rather than waiting for one that is still in use
// Size classes are powers of two (>= 32 MiB) and a request is only served by a chunk of exactly its class: every
// Metadata of a given network then draws the same multiset of classes, and the pool stops growing after the first few
// forwards.  (With best-fit over a size range, requests of concurrently building Metadata objects occasionally took each
// other's chunks and forced a cudaMalloc in steady state -- measured at 12 ms beside a busy GPU, with the driver lock
// blocking every other thread's launches.)
static size_t chunk_round(size_t b) { size_t c = 32u << 20; while (c < b) c <<= 1; return c; }
// build streams are recycled like the pinned blocks (stream creation is not free either)
static std::vector<cudaStream_t> g_stream_free, g_stream_free_lo;
static std::vector<cudaEvent_t> g_event_free;
thread_local bool tl_prefetch_worker = false;
thread_local int tl_ctx = 0; // build context of this thread: 0 = caller and chain worker, 1 = second prefetch worker
thread_local bool tl_build_here = false; // the caller's thread builds the entry itself instead of waiting for the second worker
void set_prefetch_worker_thread(bool on, int ctx) { tl_prefetch_worker = on; tl_ctx = ctx; }
// The first submanifold plan of a forward (finest grid) is on the critical path of its first convolution: the caller's
// thread, which has just built the input layer, builds it right away on the second build context instead of waiting for
// the second worker thread to wake up (measured: ~0.16 ms between the job submission and the worker's first kernel).
int build_subm_on_caller(Metadata &md, const long *sz, const long *f) {
  if (md.nCtx < 2 || tl_prefetch_worker) return 0;
  struct Scope { int old; Scope() : old(tl_ctx) { tl_ctx = 1; tl_build_here = true; } ~Scope() { tl_ctx = old; tl_build_here = false; } } scope;
  SubmEntry *e = nullptr;
  return md.get_submanifold(sz, f, &e);
}
BuildCtx &Metadata::cur() { return cx[tl_ctx < nCtx ? tl_ctx : 0]; }
Metadata::BuildLock::BuildLock(Metadata &md) : c(md.cur()) {
  if (tl_prefetch_worker) {
    while (c.callerWaiting.load(std::memory_order_acquire) > 0) std::this_thread::yield();
    c.mu.lock();
  } else {
    c.callerWaiting.fetch_add(1, std::memory_order_acq_rel);
    c.mu.lock();
    c.callerWaiting.fetch_sub(1, std::memory_order_acq_rel);
  }
}
int Metadata::mark_ready(Ready &r) {
  BuildCtx &c = cur();
  if (c.stream != cstream) {
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      if (!g_event_free.empty()) { r.ev = g_event_free.back(); g_event_free.pop_back(); }
    }
    if (!r.ev) SCN_CUDA(cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming));
    SCN_CUDA(cudaEventRecord(r.ev, c.stream));
  }
  {
    std::lock_guard<std::mutex> lk(mapMu);
    if (r.ev) events.push_back(r.ev);
    r.by = c.stream;
    r.ready = true;
    r.building = false;
  }
  cv.notify_all();
  return 0;
}
void Metadata::unclaim(Ready &r) {
  { std::lock_guard<std::mutex> lk(mapMu); r.building = false; }
  cv.notify_all();
}
bool Metadata::claim(Ready &r) {
  std::unique_lock<std::mutex> lk(mapMu);
  for (;;) {
    if (r.ready) return false;
    if (!r.building) { r.building = true; return true; }
    cv.wait(lk);
  }
}
int Metadata::need(Ready &r) {
  if (r.ev && r.by != cur().stream) SCN_CUDA(cudaStreamWaitEvent(cur().stream, r.ev, 0));
  return 0;
}
int Metadata::wait_ready(Ready &r) {
  if (r.ev && !r.waited) SCN_CUDA(cudaStreamWaitEvent(cstream, r.ev, 0));
  r.waited = true;
  return 0;
}
Metadata::~Metadata() {
  // The buffers may still be read by feature kernels queued on the caller's stream and (rarely) written by a build
  // stream: a chunk is reusable once BOTH are done.  The caller's stream is made to wait for the build streams' tails
  // and the chunks' `freed` events are recorded on the caller's stream -- the build streams themselves are never
  // blocked, so that the next Metadata (which recycles them, possibly while this forward still computes: streaming
  // inference with FPN_Net.prefetch) can start building at once.
  std::lock_guard<std::mutex> lk(g_pool_mu);
  to_compute();
  for (int i = 0; i < nCtx; i++) {
    BuildCtx &c = cx[i];
    for (Chunk &k : c.chunks) {
      if (!k.freed) cudaEventCreateWithFlags(&k.freed, cudaEventDisableTiming);
      cudaEventRecord(k.freed, cstream);
      if (g_chunk_bytes + k.cap > kChunkKeep) { cudaEventSynchronize(k.freed); cudaFree(k.p); cudaEventDestroy(k.freed); g_chunk_bytes_total -= k.cap; continue; }
      g_chunks.push_back(k);
      g_chunk_bytes += k.cap;
    }
    if (c.h_scalars) g_pinned_free.push_back(c.h_scalars);
    if (c.ownStream) (c.lowPrio ? g_stream_free_lo : g_stream_free).push_back(c.stream);
  }
  for (cudaEvent_t e : events) g_event_free.push_back(e);
  if (evCompute) cudaEventDestroy(evCompute);
}
// The build streams are high-priority so that the short build kernels of the grid pyramid get in front of the long
// convolution kernels.  A Metadata whose grids are only needed at the END of a forward (the reference-numbered twin of an
// internally numbered run) must not compete with that pyramid: its contexts move to normal-priority streams.
int Metadata::use_low_priority_streams() {
  for (int i = 0; i < nCtx; i++) {
    BuildCtx &c = cx[i];
    if (!c.ownStream || c.lowPrio) continue;
    cudaStream_t lo = nullptr;
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      if (!g_stream_free_lo.empty()) { lo = g_stream_free_lo.back(); g_stream_free_lo.pop_back(); }
    }
    if (!lo) {
      int least = 0, greatest = 0;
      SCN_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
      SCN_CUDA(cudaStreamCreateWithPriority(&lo, cudaStreamNonBlocking, least));
    }
    if (evCompute) { // what init() queued on the old stream (pool memsets) comes first
      SCN_CUDA(cudaEventRecord(evCompute, c.stream));
      SCN_CUDA(cudaStreamWaitEvent(lo, evCompute, 0));
    }
    { std::lock_guard<std::mutex> lk(g_pool_mu); g_stream_free.push_back(c.stream); }
    c.stream = lo;
    c.lowPrio = true;
  }
  return 0;
}
int Metadata::from_compute() {
  if (cur().stream == cstream || !evCompute) return 0;
  SCN_CUDA(cudaEventRecord(evCompute, cstream));
  SCN_CUDA(cudaStreamWaitEvent(cur().stream, evCompute, 0));
  return 0;
}
void Metadata::to_compute() {
  for (int i = 0; i < nCtx; i++) {
    BuildCtx &c = cx[i];
    if (evCompute && c.stream != cstream) {
      cudaEventRecord(evCompute, c.stream);
      cudaStreamWaitEvent(cstream, evCompute, 0);
    }
  }
}
void *Metadata::alloc_in(BuildCtx &c, size_t bytes) {
  void *p = nullptr;
  bytes = (std::max<size_t>(bytes, 256) + 255) & ~(size_t)255;
  if (c.arena && c.arenaUsed + bytes <= c.arenaCap) {
    p = c.arena + c.arenaUsed;
    c.arenaUsed += bytes;
    return p;
  }
  const bool dedicated = bytes > c.arenaNext / 2; // large buffers get their own block, the current chunk stays in use
  const size_t cap = chunk_round(dedicated ? bytes : c.arenaNext);
  Chunk k{nullptr, 0, nullptr};
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    // best fit among the chunks whose previous owner's work has already finished; a chunk that is still in use (its
    // forward is still computing) is taken only when the pool is full -- waiting for it would serialise this build
    // behind that forward
    int best = -1, bestBusy = -1;
    for (int i = 0; i < (int)g_chunks.size(); i++) {
      if (g_chunks[i].cap != cap) continue;
      const bool done = !g_chunks[i].freed || cudaEventQuery(g_chunks[i].freed) == cudaSuccess;
      int &b = done ? best : bestBusy;
      if (b < 0 || g_chunks[i].cap < g_chunks[b].cap) b = i;
    }
    cudaGetLastError(); // cudaEventQuery leaves cudaErrorNotReady behind
    // Nothing finished: a Metadata built AHEAD of its forward (streaming, g_pool_growth) takes fresh memory so that it does
    // not queue behind the forward that still owns the busy chunk; otherwise wait for that chunk -- a cudaMalloc beside a
    // busy GPU was measured at 0.4-100 ms and would make one-building-at-a-time latency erratic.
    if (best < 0 && bestBusy >= 0 && (!poolGrowth || g_chunk_bytes_total + cap > kChunkGrow)) { best = bestBusy; g_chunk_waits++; }
    if (best >= 0) { k = g_chunks[best]; g_chunks.erase(g_chunks.begin() + best); g_chunk_bytes -= k.cap; }
  }
  if (k.p) {
    if (cudaStreamWaitEvent(c.stream, k.freed, 0) != cudaSuccess) { set_error("cudaStreamWaitEvent failed"); return nullptr; }
  } else {
    if (cudaMalloc(&k.p, cap) != cudaSuccess) { set_error("cudaMalloc failed"); return nullptr; }
    k.cap = cap;
    { std::lock_guard<std::mutex> lk(g_pool_mu); g_chunk_bytes_total += cap; g_chunk_mallocs++; }
  }
  c.chunks.push_back(k);
  p = k.p;
  if (!dedicated) {
    c.arena = static_cast<char *>(p);
    c.arenaCap = k.cap;
    c.arenaUsed = bytes;
    c.arenaNext = std::min<size_t>(c.arenaNext * 2, 256u << 20);
  }
  return p;
}
void *Metadata::alloc(size_t bytes) { return alloc_in(cur(), bytes); }
int Metadata::init() {
  poolGrowth = g_pool_growth.load() != 0; // created ahead of its forward (FPN_Net.prefetch): see alloc_in
  static bool poolConfigured = false;
  if (!poolConfigured) {
    cudaMemPool_t pool;
    int dev = 0;
    SCN_CUDA(cudaGetDevice(&dev));
    SCN_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t thr = UINT64_MAX; // keep freed blocks cached: steady-state forwards never hit the driver
    SCN_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    poolConfigured = true;
  }
  static int async = -1, workers = -1;
  if (async < 0) {
    async = getenv("SCN_ASYNC_BUILD") ? atoi(getenv("SCN_ASYNC_BUILD")) : 1;
    workers = getenv("SCN_BUILD_WORKERS") ? atoi(getenv("SCN_BUILD_WORKERS")) : 2;
  }
  nCtx = (async && workers >= 2) ? 2 : 1;
  if (async) SCN_CUDA(cudaEventCreateWithFlags(&evCompute, cudaEventDisableTiming));
  for (int i = 0; i < nCtx; i++) {
    BuildCtx &c = cx[i];
    c.stream = cstream;
    if (async) {
      {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (!g_stream_free.empty()) { c.stream = g_stream_free.back(); g_stream_free.pop_back(); c.ownStream = true; }
      }
      if (!c.ownStream) {
        int lo = 0, hi = 0;
        SCN_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        SCN_CUDA(cudaStreamCreateWithPriority(&c.stream, cudaStreamNonBlocking, hi));
        c.ownStream = true;
      }
    }
    c.zpoolWords = 1 << 19; // 4 MiB of scan state
    c.zpool = static_cast<unsigned long long *>(alloc_in(c, c.zpoolWords * 8));
    c.d_scalars = static_cast<int *>(alloc_in(c, 256 * 4));
    SCN_CHECK(c.zpool && c.d_scalars, "alloc");
    c.d_err = c.d_scalars + 200;
    SCN_CUDA(cudaMemsetAsync(c.zpool, 0, c.zpoolWords * 8, c.stream));
    SCN_CUDA(cudaMemsetAsync(c.d_scalars, 0, 256 * 4, c.stream));
    c.h_scalars = pinned_get();
    SCN_CHECK(c.h_scalars, "pinned host scratch");
  }
  return 0;
}
unsigned long long *Metadata::scan_state(long n) {
  BuildCtx &c = cur();
  size_t w = scan_state_words(n);
  if (c.zpoolUsed + w > c.zpoolWords) { // start a fresh zeroed pool
    size_t words = std::max(c.zpoolWords, w * 2);
    c.zpool = alloc_n<unsigned long long>(words);
    if (!c.zpool) return nullptr;
    cudaMemsetAsync(c.zpool, 0, words * 8, c.stream);
    c.zpoolWords = words;
    c.zpoolUsed = 0;
  }
  unsigned long long *p = c.zpool + c.zpoolUsed;
  c.zpoolUsed += w;
  return p;
}
int Metadata::sync_scalars(int count) {
  BuildCtx &c = cur();
  SCN_CUDA(cudaMemcpyAsync(c.h_scalars, c.d_scalars, count * 4, cudaMemcpyDeviceToHost, c.stream));
  SCN_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}
// Worker threads may run ahead of the chain worker that creates the grids: wait for it.
Grid *Metadata::find_grid_wait(const long *sz) {
  std::unique_lock<std::mutex> lk(mapMu);
  for (;;) {
    auto it = grids.find(P3{sz[0], sz[1], sz[2]});
    if (it != grids.end() && it->second.built) return &it->second;
    if (!tl_prefetch_worker || chainDone.load()) return nullptr;
    cv.wait_for(lk, std::chrono::milliseconds(2));
  }
}
ConvEntry *Metadata::wait_conv(const long *inS, const long *f, const long *st) {
  ConvKey key{P3{inS[0], inS[1], inS[2]}, P3{f[0], f[1], f[2]}, P3{st[0], st[1], st[2]}};
  std::unique_lock<std::mutex> lk(mapMu);
  for (;;) {
    auto it = conv.find(key);
    if (it != conv.end() && it->second.rdy.ready) return &it->second;
    if (chainDone.load()) return nullptr;
    cv.wait_for(lk, std::chrono::milliseconds(2));
  }
}
void Metadata::set_chain_done(bool v) {
  chainDone.store(v);
  cv.notify_all();
}
Grid *Metadata::find_grid(const long *sz) {
  std::lock_guard<std::mutex> lk(mapMu);
  auto it = grids.find(P3{sz[0], sz[1], sz[2]});
  return it == grids.end() || !it->second.built ? nullptr : &it->second;
}

template <class InF, class OutF>
static int run_scan(Metadata &M, long n, InF in, OutF out, int *total) {
  if (n <= 0) {
    if (total) SCN_CUDA(cudaMemsetAsync(total, 0, 4, M.cur().stream));
    return 0;
  }
  unsigned long long *st = M.scan_state(n);
  SCN_CHECK(st, "scan state");
  scan_kernel<<<cdiv(n, kScanTile), kScanThreads, 0, LS(M.cur().stream)>>>(n, in, out, st, total);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

static GridView view(const Grid &g) {
  return GridView{g.dir, g.bmask, g.wbase, g.dd[0], g.dd[1], g.dd[2], g.dirCells, (int)g.sz[0], (int)g.sz[1], (int)g.sz[2]};
}

// ------------------------------------------------------------------ block structure
__global__ void k_coords_to_pts(const long *coords, long n, int ncols, int4 *pts, int *maxBatch) {
  int mb = 0;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const long *c = coords + i * ncols;
    int b = ncols == 4 ? (int)c[3] : 0;
    pts[i] = make_int4((int)c[0], (int)c[1], (int)c[2], b);
    mb = max(mb, b);
  }
  if (ncols == 4) {
    for (int d = 16; d > 0; d >>= 1) mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, d));
    if ((threadIdx.x & 31) == 0 && mb > 0) atomicMax(maxBatch, mb);
  }
}
__device__ __forceinline__ long dir_cell(const int4 &p, int dd1, int dd2, long dirCells) {
  return (long)p.w * dirCells + ((long)(p.x >> 3) * dd1 + (p.y >> 3)) * dd2 + (p.z >> 3);
}
__global__ void k_mark_dir(const int4 *pts, long n, int *dir, int dd1, int dd2, long dirCells, int sz0, int sz1, int sz2, int *err) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int4 p = pts[i];
    if (p.x < 0) continue; // invalid event
    if (p.x >= sz0 || (unsigned)p.y >= (unsigned)sz1 || (unsigned)p.z >= (unsigned)sz2) { *err = 2; continue; }
    dir[dir_cell(p, dd1, dd2, dirCells)] = 1;
  }
}
struct DirIn { const int *dir; __device__ int operator()(long i) const { return dir[i] != 0; } };
struct DirOut { int *dir; __device__ void operator()(long i, int pre, int v) const { dir[i] = v ? pre : -1; } };
__global__ void k_zero_words(unsigned long long *w, const int *nblocks) {
  long n = (long)(*nblocks) * 8;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) w[i] = 0ull;
}
__global__ void k_set_bits(const int4 *pts, long n, const int *dir, unsigned long long *bmask, int dd1, int dd2, long dirCells, int sz0, int sz1, int sz2) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int4 p = pts[i];
    if (p.x < 0 || p.x >= sz0 || (unsigned)p.y >= (unsigned)sz1 || (unsigned)p.z >= (unsigned)sz2) continue;
    int blk = dir[dir_cell(p, dd1, dd2, dirCells)];
    int bit = ((p.x & 7) << 6) | ((p.y & 7) << 3) | (p.z & 7);
    atomicOr(bmask + (long)blk * 8 + (bit >> 6), 1ull << (bit & 63));
  }
}
struct WordIn {
  const unsigned long long *bmask; const int *nblocks;
  __device__ int operator()(long i) const { return i < (long)(*nblocks) * 8 ? __popcll(bmask[i]) : 0; }
};
struct WordOut {
  int *wbase; const int *nblocks;
  __device__ void operator()(long i, int pre, int) const { if (i < (long)(*nblocks) * 8) wbase[i] = pre; }
};
__global__ void k_lookup_pts(GridView g, const int4 *pts, long n, int *outP) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int4 p = pts[i];
    outP[i] = p.x < 0 ? -1 : grid_lookup(g, p.x, p.y, p.z, p.w);
  }
}

// Builds dir / bmask / wbase of `g` from a point list (duplicates and x<0 "invalid" entries
// allowed); d_nunique receives the number of distinct points; outP[i] = spatial index of pts[i].
static int build_blocks(Metadata &M, Grid &g, const int4 *pts, long npts, int *outP, int *d_nunique) {
  for (int d = 0; d < 3; d++) g.dd[d] = (int)((g.sz[d] + 7) / 8);
  g.dirCells = (long)g.dd[0] * g.dd[1] * g.dd[2];
  long cells = g.dirCells * g.batch;
  SCN_CHECK(cells < (1l << 30), "spatial size too large for the block directory");
  g.dir = M.alloc_n<int>(cells);
  g.d_nblocks = M.alloc_n<int>(4);
  g.maxBlocks = std::max(1l, std::min(npts, cells));
  g.bmask = M.alloc_n<unsigned long long>(g.maxBlocks * 8);
  g.wbase = M.alloc_n<int>(g.maxBlocks * 8);
  SCN_CHECK(g.dir && g.bmask && g.wbase && g.d_nblocks, "alloc");
  cudaStream_t s = M.cur().stream;
  SCN_CUDA(cudaMemsetAsync(g.dir, 0, cells * 4, s));
  if (npts > 0) {
    k_mark_dir<<<stream_grid(npts, 256), 256, 0, LS(s)>>>(pts, npts, g.dir, g.dd[1], g.dd[2], g.dirCells, (int)g.sz[0], (int)g.sz[1], (int)g.sz[2], M.cur().d_err);
  }
  SCN_TRY(run_scan(M, cells, DirIn{g.dir}, DirOut{g.dir}, g.d_nblocks));
  k_zero_words<<<stream_grid(g.maxBlocks * 8, 256), 256, 0, LS(s)>>>(g.bmask, g.d_nblocks);
  if (npts > 0) {
    k_set_bits<<<stream_grid(npts, 256), 256, 0, LS(s)>>>(pts, npts, g.dir, g.bmask, g.dd[1], g.dd[2], g.dirCells, (int)g.sz[0], (int)g.sz[1], (int)g.sz[2]);
  }
  SCN_TRY(run_scan(M, g.maxBlocks * 8, WordIn{g.bmask, g.d_nblocks}, WordOut{g.wbase, g.d_nblocks}, d_nunique));
  if (npts > 0 && outP) k_lookup_pts<<<stream_grid(npts, 256), 256, 0, LS(s)>>>(view(g), pts, npts, outP);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ input layer
__global__ void k_fill_int(int *p, long n, int v) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void k_first_rows(const int *rowP, long n, int *firstRow, int *lastRow, int *cnt, int *maxCnt) {
  int mc = 0;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int p = rowP[i];
    atomicMin(firstRow + p, (int)i);
    if (lastRow) atomicMax(lastRow + p, (int)i);
    int c = atomicAdd(cnt + p, 1) + 1;
    mc = max(mc, c);
  }
  for (int d = 16; d > 0; d >>= 1) mc = max(mc, __shfl_xor_sync(0xffffffffu, mc, d));
  if ((threadIdx.x & 31) == 0 && mc > 0) atomicMax(maxCnt, mc);
}
struct FirstIn {
  const int *rowP, *firstRow;
  __device__ int operator()(long i) const { return firstRow[rowP[i]] == (int)i; }
};
struct FirstOut {
  const int *rowP; const int4 *pts; int *p2id, *id2p; int4 *coords;
  __device__ void operator()(long i, int pre, int v) const {
    if (v) { int p = rowP[i]; p2id[p] = pre; id2p[pre] = p; coords[pre] = pts[i]; }
  }
};
// rules table rows: [count, rows ascending..., 0 padding]  (IOLayersRules.h:111-124)
__global__ void k_input_rules_fill(const int *rowP, const int *p2id, long n, int *tab, int w) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int id = p2id[rowP[i]];
    int slot = atomicAdd(tab + (long)id * w, 1);
    tab[(long)id * w + 1 + slot] = (int)i;
  }
}
__global__ void k_input_rules_sort(int *tab, int nOut, int w) {
  for (long id = blockIdx.x * (long)blockDim.x + threadIdx.x; id < nOut; id += (long)gridDim.x * blockDim.x) {
    int *r = tab + id * w;
    int c = r[0];
    for (int a = 2; a <= c; a++) { // insertion sort, lists are tiny
      int v = r[a], b = a - 1;
      while (b >= 1 && r[b] > v) { r[b + 1] = r[b]; b--; }
      r[b + 1] = v;
    }
  }
}
__global__ void k_input_rules_pick(const int *pick, const int *id2p, int nOut, int *tab) {
  for (long id = blockIdx.x * (long)blockDim.x + threadIdx.x; id < nOut; id += (long)gridDim.x * blockDim.x) {
    tab[id * 2] = 1;
    tab[id * 2 + 1] = pick[id2p[id]];
  }
}
__global__ void k_count_batch(const int4 *coords, int n, int *counts) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) atomicAdd(counts + coords[i].w, 1);
}

__global__ void k_iota(int *p, int n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = (int)i;
}
// spatialIds: row id = spatial index.  One writer per site (the first input row / any event of the site: same values).
__global__ void k_spatial_input_ids(const int *rowP, const int4 *pts, long n, const int *firstRow, int4 *coords, int *p2id, int *id2p) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int p = rowP[i];
    if (firstRow[p] == (int)i) { coords[p] = pts[i]; p2id[p] = p; id2p[p] = p; }
  }
}
__global__ void k_spatial_conv_ids(const int *evQ, const int4 *evPts, long E, int4 *coords, int *p2id, int *id2p) {
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < E; e += (long)gridDim.x * blockDim.x) {
    const int q = evQ[e];
    if (q >= 0) { coords[q] = evPts[e]; p2id[q] = q; id2p[q] = q; }
  }
}
__global__ void k_copy_scalar(const int *src, int *dst) { *dst = *src; }

// Metadata::inputLayer -> inputLayerRules (SCN/Metadata/Metadata.cpp:405-417, IOLayersRules.h:18-125).
int Metadata::input_layer(const long *sz, const long *coords, int onDevice, long nrows, int ncols, int batchHint, int mode) {
  SCN_CHECK(ncols == 3 || ncols == 4, "coords must be N x 3 or N x 4");
  SCN_CHECK(mode >= 0 && mode <= 4, "mode");
  SCN_CHECK(nrows < (1l << 26), "too many input rows");
  P3 key{sz[0], sz[1], sz[2]};
  BuildLock bl(*this);
  Grid *gp;
  {
    std::lock_guard<std::mutex> lk(mapMu);
    SCN_CHECK(grids.find(key) == grids.end() && !input.valid, "input layer already built for this Metadata");
    gp = &grids[key];
  }
  Grid &g = *gp;
  g.sz = key;
  cudaStream_t s = cur().stream;
  if (onDevice == 1) SCN_TRY(from_compute()); // the coordinates were produced on the caller's stream (2: already complete, no dependency)
  const long *dcoords = coords;
  if (!onDevice && nrows) {
    long *tmp = alloc_n<long>(nrows * ncols);
    SCN_CHECK(tmp, "alloc");
    SCN_CUDA(cudaMemcpyAsync(tmp, coords, nrows * ncols * 8, cudaMemcpyHostToDevice, s));
    ++g_counters[kCntCoordUpload];
    dcoords = tmp;
  }
  int4 *pts = alloc_n<int4>(std::max(1l, nrows));
  SCN_CHECK(pts, "alloc");
  int *sc = cur().d_scalars; // [0] maxBatch [1] nUnique [2] maxActive [3] nActive
  SCN_CUDA(cudaMemsetAsync(sc, 0, 64 * 4, s));
  if (nrows) k_coords_to_pts<<<stream_grid(nrows, 256), 256, 0, LS(s)>>>(dcoords, nrows, ncols, pts, sc);
  g.batch = std::max(1, batchHint);
  if (ncols == 4 && nrows) {
    SCN_TRY(sync_scalars(1));
    g.batch = std::max(g.batch, cur().h_scalars[0] + 1);
  }
  SCN_CHECK(g.batch <= 48, "batch size > 48 not supported");
  int *rowP = alloc_n<int>(std::max(1l, nrows));
  SCN_TRY(build_blocks(*this, g, pts, nrows, rowP, sc + 1));
  long cap = std::max(1l, nrows);
  g.coords = alloc_n<int4>(cap);
  g.p2id = alloc_n<int>(cap);
  g.id2p = alloc_n<int>(cap);
  int *firstRow = alloc_n<int>(cap), *cnt = alloc_n<int>(cap), *lastRow = mode == 2 ? alloc_n<int>(cap) : nullptr;
  SCN_CHECK(g.coords && g.p2id && g.id2p && firstRow && cnt, "alloc");
  SCN_CUDA(cudaMemsetAsync(firstRow, 0x7f, cap * 4, s));
  SCN_CUDA(cudaMemsetAsync(cnt, 0, cap * 4, s));
  if (lastRow) SCN_CUDA(cudaMemsetAsync(lastRow, 0xff, cap * 4, s));
  if (nrows) k_first_rows<<<stream_grid(nrows, 256), 256, 0, LS(s)>>>(rowP, nrows, firstRow, lastRow, cnt, sc + 2);
  if (spatialIds) {
    if (nrows) k_spatial_input_ids<<<stream_grid(nrows, 256), 256, 0, LS(s)>>>(rowP, pts, nrows, firstRow, g.coords, g.p2id, g.id2p);
    k_copy_scalar<<<1, 1, 0, LS(s)>>>(sc + 1, sc + 3); // nActive = number of distinct sites
  } else {
    SCN_TRY(run_scan(*this, nrows, FirstIn{rowP, firstRow}, FirstOut{rowP, pts, g.p2id, g.id2p, g.coords}, sc + 3));
  }
  // per-batch-item counts (only needed when batch > 1)
  SCN_TRY(sync_scalars(4));
  g.n = cur().h_scalars[3];
  int maxActive = cur().h_scalars[2];
  SCN_CHECK(cur().h_scalars[1] == g.n, "internal: unique count mismatch");
  g.itemCount.assign(g.batch, 0);
  g.itemCtr.assign(g.batch, g.batch == 1 ? 0 : -1);
  if (g.batch == 1) g.itemCount[0] = g.n;
  else {
    SCN_CUDA(cudaMemsetAsync(sc + 8, 0, 48 * 4, s));
    if (g.n) k_count_batch<<<stream_grid(g.n, 256), 256, 0, LS(s)>>>(g.coords, g.n, sc + 8);
    SCN_TRY(sync_scalars(8 + 48));
    for (int b = 0; b < g.batch; b++) g.itemCount[b] = cur().h_scalars[8 + b];
  }
  { std::lock_guard<std::mutex> lk(mapMu); g.built = true; }
  SCN_TRY(mark_ready(g.rdy));
  input.mode = mode; input.nIn = (int)nrows; input.nOut = g.n; input.valid = true;
  input.maxActive = (mode == 3 || mode == 4) ? maxActive : 1;
  input.rowP = rowP; input.firstRow = firstRow; input.lastRow = lastRow; input.pts = pts;
  return input_rules(g);
}
// The rule table of the input layer in the numbering of g (input.mode / maxActive / nIn / rowP / firstRow / lastRow are set).
int Metadata::input_rules(const Grid &g) {
  if (input.mode == 0) { input.tab = nullptr; return mark_ready(input.rdy); }
  cudaStream_t s = cur().stream;
  int w = 1 + input.maxActive;
  input.tab = alloc_n<int>(std::max(1l, (long)g.n * w));
  SCN_CHECK(input.tab, "alloc");
  if (g.n == 0) return mark_ready(input.rdy);
  if (input.mode == 3 || input.mode == 4) {
    SCN_CUDA(cudaMemsetAsync(input.tab, 0, (long)g.n * w * 4, s));
    k_input_rules_fill<<<stream_grid(input.nIn, 256), 256, 0, LS(s)>>>(input.rowP, g.p2id, input.nIn, input.tab, w);
    if (input.maxActive > 1) k_input_rules_sort<<<stream_grid(g.n, 256), 256, 0, LS(s)>>>(input.tab, g.n, w);
  } else {
    // IOLayersRules.h:100-110: mode 1 keeps the FIRST row of a voxel, mode 2 the LAST
    k_input_rules_pick<<<stream_grid(g.n, 256), 256, 0, LS(s)>>>(input.mode == 1 ? input.firstRow : input.lastRow, g.id2p, g.n, input.tab);
  }
  SCN_CUDA(cudaGetLastError());
  return mark_ready(input.rdy);
}

// ------------------------------------------------------------------ numbering overlay
// copies the block structure of `src` (same spatial size and sites) into g's own buffers; only the nblocks * 8 live occupancy
// words are copied -- maxBlocks is bounded by the input rows, at level 0 many times the live blocks
__global__ void k_copy_words(const unsigned long long *__restrict__ bmask, const int *__restrict__ wbase, const int *__restrict__ nblocks,
                             unsigned long long *__restrict__ bOut, int *__restrict__ wOut) {
  const long n = (long)(*nblocks) * 8;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) { bOut[i] = bmask[i]; wOut[i] = wbase[i]; }
}
static int copy_blocks(Metadata &M, Grid &g, const Grid &src) {
  for (int d = 0; d < 3; d++) g.dd[d] = src.dd[d];
  g.dirCells = src.dirCells;
  g.maxBlocks = src.maxBlocks;
  const long cells = g.dirCells * g.batch;
  g.dir = M.alloc_n<int>(cells);
  g.d_nblocks = M.alloc_n<int>(4);
  g.bmask = M.alloc_n<unsigned long long>(g.maxBlocks * 8);
  g.wbase = M.alloc_n<int>(g.maxBlocks * 8);
  SCN_CHECK(g.dir && g.bmask && g.wbase && g.d_nblocks, "alloc");
  cudaStream_t s = M.cur().stream;
  SCN_CUDA(cudaMemcpyAsync(g.dir, src.dir, cells * 4, cudaMemcpyDeviceToDevice, s));
  SCN_CUDA(cudaMemcpyAsync(g.d_nblocks, src.d_nblocks, 4, cudaMemcpyDeviceToDevice, s));
  k_copy_words<<<stream_grid(g.maxBlocks * 8, 256), 256, 0, LS(s)>>>(src.bmask, src.wbase, src.d_nblocks, g.bmask, g.wbase);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
// The internally numbered grid of size sz once `in`'s chain worker has made it (nullptr: the chain worker has finished without it);
// this build stream waits for it.
static Grid *internal_grid(Metadata &M, Metadata &in, const long *sz) {
  Grid *gq = in.find_grid_wait(sz);
  if (gq && gq->rdy.ev && cudaStreamWaitEvent(M.cur().stream, gq->rdy.ev, 0) != cudaSuccess) return nullptr;
  return gq;
}
static Grid *new_grid(Metadata &M, const long *sz) {
  std::lock_guard<std::mutex> lk(M.mapMu);
  const P3 key{sz[0], sz[1], sz[2]};
  if (M.grids.find(key) != M.grids.end()) return nullptr;
  Grid *g = &M.grids[key];
  g->sz = key;
  return g;
}
static int publish_grid(Metadata &M, Grid &g) {
  g.itemCount.assign(1, g.n);
  g.itemCtr.assign(1, 0);
  SCN_TRY(M.mark_ready(g.rdy)); // the event first: a thread that sees `built` must also see the event to wait for
  { std::lock_guard<std::mutex> lk(M.mapMu); g.built = true; }
  M.cv.notify_all();
  return 0;
}
// Input level: the reference id of a site is the rank of its first input row among the first rows of all sites (FirstIn /
// FirstOut, as in input_layer), read from the internal input layer's arrays -- no coordinate upload, no block build.
int Metadata::overlay_input(Metadata &in, const long *sz) {
  Grid *gq = in.find_grid(sz);
  SCN_CHECK(gq && in.input.valid && gq->batch == 1, "numbering overlay: the internal input layer is missing");
  BuildLock bl(*this);
  SCN_CHECK(!input.valid, "input layer already built for this Metadata");
  Grid *gp = new_grid(*this, sz);
  SCN_CHECK(gp, "input layer already built for this Metadata");
  Grid &g = *gp;
  cudaStream_t s = cur().stream;
  if (gq->rdy.ev) SCN_CUDA(cudaStreamWaitEvent(s, gq->rdy.ev, 0));
  g.batch = 1;
  g.n = gq->n;
  SCN_TRY(copy_blocks(*this, g, *gq));
  const long nrows = in.input.nIn, cap = std::max(1, g.n);
  g.coords = alloc_n<int4>(cap);
  g.p2id = alloc_n<int>(cap);
  g.id2p = alloc_n<int>(cap);
  SCN_CHECK(g.coords && g.p2id && g.id2p, "alloc");
  const InputRules &I = in.input;
  SCN_TRY(run_scan(*this, nrows, FirstIn{I.rowP, I.firstRow}, FirstOut{I.rowP, I.pts, g.p2id, g.id2p, g.coords}, nullptr));
  SCN_TRY(publish_grid(*this, g));
  input.mode = I.mode; input.nIn = I.nIn; input.nOut = g.n; input.maxActive = I.maxActive; input.valid = true;
  input.rowP = I.rowP; input.firstRow = I.firstRow; input.lastRow = I.lastRow; input.pts = I.pts;
  SCN_TRY(input_rules(g));
  input.rowP = input.firstRow = input.lastRow = nullptr; // `in`'s buffers: not kept beyond this build
  input.pts = nullptr;
  return 0;
}

// ------------------------------------------------------------------ dense_hash_map order
// Emulates the bucket layout google::dense_hash_map reaches when the keys are inserted one by one
// (growth by doubling at load 0.5, re-insertion in ascending bucket order, triangular probing).
// Table entry (32 bit): [31:7] insertion rank within the current growth phase | [6:0] probe count.
// Lower rank wins a bucket; the row id of rank r is seq[r].
constexpr unsigned kEmpty = 0xffffffffu;
constexpr unsigned kProbeBits = 7, kProbeMask = (1u << kProbeBits) - 1u;
// Priority insertion: the key of insertion rank i must end at the first bucket of its probe path
// (b, b+1, b+3, b+6, ...) that no lower-ranked key occupies -- exactly what sequential insertion
// produces.  A displaced key is carried onwards by the displacing thread; its next bucket follows
// from the bucket it sat in and its stored probe count, so its hash is not needed again.
__device__ __forceinline__ void priority_insert(unsigned *tab, unsigned mask, unsigned b, unsigned cur, int *err) {
  while (true) {
    unsigned old = atomicMin(tab + b, cur);
    if (old == kEmpty) return;
    if (old > cur) cur = old;
    unsigned probe = (cur & kProbeMask) + 1u;
    if (probe > kProbeMask) { *err = 3; return; }
    cur = (cur & ~kProbeMask) | probe;
    b = (b + probe) & mask;
  }
}
struct TabIn { const unsigned *tab; __device__ int operator()(long i) const { return tab[i] != kEmpty; } };
// ids of the old table's elements in ascending bucket order (the re-insertion order on growth)
struct CompactOut {
  const unsigned *tab; const int *seqIn; int idOffset; int *seqOut;
  __device__ void operator()(long i, int pre, int v) const {
    if (v) { unsigned r = tab[i] >> kProbeBits; seqOut[pre] = seqIn ? seqIn[r] : (int)r + idOffset; }
  }
};
// one thread per key: ranks [0, nPrev) are the re-inserted old keys (ids in oldSeq), ranks
// [nPrev, nCur) the keys inserted during this phase (ids newSeq[rank] or rank + idOffset)
__global__ void __launch_bounds__(256) k_phase_insert(unsigned *cur, unsigned mask, const int4 *__restrict__ coords, const int *oldSeq,
                                                      const int *newSeq, int idOffset, int nPrev, int nCur, int *phaseSeq, int *err) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nCur; j += gridDim.x * blockDim.x) {
    int id = j < nPrev ? oldSeq[j] : (newSeq ? newSeq[j] : j + idOffset);
    if (phaseSeq) phaseSeq[j] = id;
    int4 c = coords[id];
    priority_insert(cur, mask, point_hash(c.x, c.y, c.z) & mask, (unsigned)j << kProbeBits, err);
  }
}
struct PhaseIn {
  const unsigned *tab; long nbPrev;
  __device__ int operator()(long i) const { return i < nbPrev && tab[i] != kEmpty; }
};
struct PhaseOut {
  const unsigned *tab; long nbPrev; const int *seqIn, *newSeq; int idOffset, nPrev; int *seqOut; unsigned *cur; unsigned mask; const int4 *coords; int *err;
  __device__ void operator()(long i, int pre, int v) const {
    int j, id;
    if (i < nbPrev) {
      if (!v) return;
      id = seqIn[tab[i] >> kProbeBits];
      j = pre;
    } else {
      j = nPrev + (int)(i - nbPrev);
      id = newSeq ? newSeq[j] : j + idOffset;
    }
    seqOut[j] = id;
    const int4 c = coords[id];
    priority_insert(cur, mask, point_hash(c.x, c.y, c.z) & mask, (unsigned)j << kProbeBits, err);
  }
};
struct OrderOut {
  const unsigned *tab; const int *seq; int *rank2id;
  __device__ void operator()(long i, int pre, int v) const { if (v) rank2id[pre] = seq[tab[i] >> kProbeBits]; }
};

// The first growth phases (tables up to kSmallNb buckets) in one CTA, entirely in shared memory.
// Leaves the last small table in `out` and the id of every rank of that phase in `seqOut`.
constexpr int kSmallNb = 16384;
struct SmallEmu { unsigned *tab; int *seq; int nb, nCur; }; // last table the CTA built (shared memory), rank -> id of that phase
// cap = buckets of the largest table this call can reach (a power of two <= kSmallNb): shared memory = 3 * cap words
__device__ __forceinline__ SmallEmu emulate_small_body(const int4 *coords, const int *seq, int idOffset, int n, unsigned *sm, int cap, int *err) {
  unsigned *A = sm, *B = sm + cap;
  int *seqA = reinterpret_cast<int *>(sm + 2 * cap), *seqB = seqA + cap / 2; // rank -> id of the two live phases
  __shared__ int s_scan[1024 / 32];
  __shared__ int s_carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  unsigned *prev = A, *cur = B;
  int *seqPrev = seqA, *seqCur = seqB;
  int nb = 32, nPrev = 0;
  while (true) {
    const int nCur = min(n, nb / 2);
    const unsigned mask = nb - 1;
    for (int i = tid; i < nb; i += 1024) cur[i] = kEmpty;
    __syncthreads();
    if (nPrev > 0) { // old elements in ascending bucket order of prev (rank = prefix count)
      const int nbPrev = nb / 2;
      if (tid == 0) s_carry = 0;
      __syncthreads();
      for (int base = 0; base < nbPrev; base += 1024) {
        int i = base + tid;
        unsigned e = i < nbPrev ? prev[i] : kEmpty;
        int v = e != kEmpty;
        int incl = warp_incl_scan(v, lane);
        if (lane == 31) s_scan[wid] = incl;
        __syncthreads();
        if (wid == 0) { int w = s_scan[lane]; int wi = warp_incl_scan(w, lane); s_scan[lane] = wi - w; }
        __syncthreads();
        int rank = s_carry + s_scan[wid] + incl - v;
        if (v) {
          int id = seqPrev[e >> kProbeBits];
          seqCur[rank] = id;
          int4 c = coords[id];
          priority_insert(cur, mask, point_hash(c.x, c.y, c.z) & mask, (unsigned)rank << kProbeBits, err);
        }
        __syncthreads();
        if (tid == 1023) s_carry = rank + v;
        __syncthreads();
      }
    }
    for (int j = nPrev + tid; j < nCur; j += 1024) {
      int id = seq ? seq[j] : j + idOffset;
      seqCur[j] = id;
      int4 c = coords[id];
      priority_insert(cur, mask, point_hash(c.x, c.y, c.z) & mask, (unsigned)j << kProbeBits, err);
    }
    __syncthreads();
    if (nCur == n || nb == cap) return SmallEmu{cur, seqCur, nb, nCur};
    unsigned *t = prev; prev = cur; cur = t;
    int *ts = seqPrev; seqPrev = seqCur; seqCur = ts;
    nPrev = nCur;
    nb *= 2;
  }
}
__global__ void __launch_bounds__(1024) k_emulate_small(const int4 *coords, const int *seq, int idOffset, int n, int cap, unsigned *out, int *seqOut, int *err) {
  extern __shared__ unsigned sm[];
  const SmallEmu e = emulate_small_body(coords, seq, idOffset, n, sm, cap, err);
  for (int i = threadIdx.x; i < e.nb; i += 1024) out[i] = e.tab[i];
  for (int i = threadIdx.x; i < e.nCur; i += 1024) seqOut[i] = e.seq[i];
}

// Hash-iteration order of one batch item: ids seq[0..n) (or idOffset + 0..n) inserted in that order.
static int emulate_order(Metadata &M, const int4 *coords, const int *seq, int idOffset, int n, int *rank2idOut) {
  if (n == 0) return 0;
  SCN_CHECK(n < (1 << 25), "too many active sites in one batch item for the hash-order emulation");
  cudaStream_t s = M.cur().stream;
  long nbFinal = 32;
  while (n > nbFinal / 2) nbFinal *= 2;
  int *S0 = M.alloc_n<int>(n), *S1 = M.alloc_n<int>(n);
  const int cap = (int)std::min<long>(nbFinal, kSmallNb);
  // one table per growth phase beyond the small ones (cap*2, cap*4, ..., nbFinal buckets: < 2 nbFinal words in all),
  // cleared by ONE memset up front, so that a phase is a single launch
  unsigned *T0 = M.alloc_n<unsigned>(cap), *big = nbFinal > cap ? M.alloc_n<unsigned>(2 * nbFinal) : nullptr;
  SCN_CHECK(T0 && S0 && S1 && (big || nbFinal <= cap), "alloc");
  if (big) SCN_CUDA(cudaMemsetAsync(big, 0xff, (size_t)(2 * nbFinal - 2 * cap) * 4, s));
  const int smallSmem = 3 * cap * 4; // small grids leave shared memory to whatever else runs on that SM
  static bool attr = false;
  if (!attr) {
    SCN_CUDA(cudaFuncSetAttribute(k_emulate_small, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * kSmallNb * 4));
    attr = true;
  }
  k_emulate_small<<<1, 1024, smallSmem, LS(s)>>>(coords, seq, idOffset, n, cap, T0, S0, M.cur().d_err);
  SCN_CUDA(cudaGetLastError());
  long nb = cap;
  unsigned *prev = T0, *cur = big;
  int *seqPrev = S0, *seqCur = S1; // seqPrev: rank -> id of the phase held in `prev`
  int nPrev = (int)std::min<long>(n, nb / 2);
  static int fusedPhases = -1;
  if (fusedPhases < 0) fusedPhases = getenv("SCN_PHASE_FUSED") ? atoi(getenv("SCN_PHASE_FUSED")) : 0; // measured: the fused launch is 2x slower (8 sequential insertions per scan thread)
  while (nb < nbFinal) {
    const long nbPrev = nb;
    nb *= 2;
    int nCur = (int)std::min<long>(n, nb / 2);
    if (!fusedPhases) { // two launches: compaction scan, then one thread per key
      SCN_TRY(run_scan(M, nbPrev, TabIn{prev}, CompactOut{prev, seqPrev, 0, seqCur}, nullptr));
      k_phase_insert<<<stream_grid(nCur, 256, 16), 256, 0, LS(s)>>>(cur, (unsigned)(nb - 1), coords, seqCur, seq, idOffset, nPrev, nCur, seqCur, M.cur().d_err);
      prev = cur; cur += nb; std::swap(seqPrev, seqCur); nPrev = nCur;
      continue;
    }
    // One launch per phase: a scan over the old table ranks its keys in ascending bucket order and its consumer
    // inserts them straight away; the keys that arrive during this phase (ranks nPrev..nCur) ride along as extra
    // scan items with value 0 -- priority insertion reaches the same fixed point in any order.
    SCN_TRY(run_scan(M, nbPrev + (nCur - nPrev), PhaseIn{prev, nbPrev},
                     PhaseOut{prev, nbPrev, seqPrev, seq, idOffset, nPrev, seqCur, cur, (unsigned)(nb - 1), coords, M.cur().d_err}, nullptr));
    prev = cur;
    cur += nb;
    std::swap(seqPrev, seqCur);
    nPrev = nCur;
  }
  SCN_TRY(run_scan(M, nbFinal, TabIn{prev}, OrderOut{prev, seqPrev, rank2idOut}, nullptr));
  SCN_CUDA(cudaGetLastError());
  return 0;
}

struct BatchIn { const int4 *coords; int b; __device__ int operator()(long i) const { return coords[i].w == b; } };
struct BatchOut { int *seq; __device__ void operator()(long i, int pre, int v) const { if (v) seq[pre] = (int)i; } };

int Metadata::ensure_rank(Grid &g) {
  if (!claim(g.rankRdy)) return need(g.rankRdy); // built by another thread, possibly on the other build stream
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, g.rankRdy};
  SCN_TRY(need(g.rdy)); // (every caller already holds the lock of its build context)
  g.rank2id = alloc_n<int>(std::max(1, g.n));
  SCN_CHECK(g.rank2id, "alloc");
  if (spatialIds) { // sites are visited in row order: no hash-order emulation
    if (g.n) k_iota<<<stream_grid(g.n, 256), 256, 0, LS(cur().stream)>>>(g.rank2id, g.n);
    g.hasRank = true;
    return mark_ready(g.rankRdy);
  }
  int start = 0;
  for (int b = 0; b < g.batch; b++) {
    int cnt = g.itemCount[b];
    if (g.itemCtr[b] >= 0) {
      SCN_TRY(emulate_order(*this, g.coords, nullptr, g.itemCtr[b], cnt, g.rank2id + start));
    } else { // ids of item b interleave with other items: compact them in ascending id order
      int *seq = alloc_n<int>(std::max(1, cnt));
      SCN_CHECK(seq, "alloc");
      SCN_TRY(run_scan(*this, g.n, BatchIn{g.coords, b}, BatchOut{seq}, nullptr));
      SCN_TRY(emulate_order(*this, g.coords, seq, 0, cnt, g.rank2id + start));
    }
    start += cnt;
  }
  g.hasRank = true;
  return mark_ready(g.rankRdy);
}

// ------------------------------------------------------------------ rule lists (shared machinery)
// Events are visited in reference order (rank-major).  Each rank r owns at most one event per
// list, so the position of (r, L) inside list L is the number of earlier ranks with an event in L.
constexpr int kRuleTile = 256;
__device__ __forceinline__ void tile_list_counts(unsigned long long mask, int K, int (*s_cnt)[64], int lane, int wid) {
  for (int L = 0; L < K; L++) {
    unsigned bal = __ballot_sync(0xffffffffu, (mask >> L) & 1ull);
    if (lane == 0) s_cnt[wid][L] = __popc(bal);
  }
}
// tileCnt[tile*K + L]
template <class MaskF>
__global__ void __launch_bounds__(kRuleTile) k_rule_count(int n, int K, MaskF maskf, int *tileCnt) {
  __shared__ int s_cnt[kRuleTile / 32][64];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int r = blockIdx.x * kRuleTile + tid;
  unsigned long long mask = r < n ? maskf(r) : 0ull;
  tile_list_counts(mask, K, s_cnt, lane, wid);
  __syncthreads();
  if (tid < K) {
    int c = 0;
    for (int w = 0; w < kRuleTile / 32; w++) c += s_cnt[w][tid];
    tileCnt[(long)blockIdx.x * K + tid] = c;
  }
}
// one CTA per list: exclusive scan of tileCnt[., L] over tiles (in place), totals[L]
__global__ void __launch_bounds__(1024) k_rule_scan(int nTiles, int K, int *tileCnt, int *totals) {
  __shared__ int s_scan[32];
  __shared__ int s_carry;
  const int L = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < nTiles; base += 1024) {
    int i = base + tid;
    int v = i < nTiles ? tileCnt[(long)i * K + L] : 0;
    int incl = warp_incl_scan(v, lane);
    if (lane == 31) s_scan[wid] = incl;
    __syncthreads();
    if (wid == 0) { int w = s_scan[lane]; int wi = warp_incl_scan(w, lane); s_scan[lane] = wi - w; }
    __syncthreads();
    int ex = s_carry + s_scan[wid] + incl - v;
    if (i < nTiles) tileCnt[(long)i * K + L] = ex;
    __syncthreads();
    if (tid == 1023) s_carry = ex + v;
    __syncthreads();
  }
  if (tid == 0) totals[L] = s_carry;
}
__global__ void k_list_offsets(int K, const int *totals, int *off) {
  if (threadIdx.x == 0) { int a = 0; for (int L = 0; L < K; L++) { off[L] = a; a += totals[L]; } off[K] = a; }
}
template <class MaskF, class PairF>
__global__ void __launch_bounds__(kRuleTile) k_rule_write(int n, int K, MaskF maskf, PairF pairf, const int *tileBase, const int *off, int2 *pairs) {
  __shared__ int s_cnt[kRuleTile / 32][64];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int r = blockIdx.x * kRuleTile + tid;
  unsigned long long mask = r < n ? maskf(r) : 0ull;
  tile_list_counts(mask, K, s_cnt, lane, wid);
  __syncthreads();
  if (tid < K) { // exclusive prefix over warps
    int a = 0;
    for (int w = 0; w < kRuleTile / 32; w++) { int c = s_cnt[w][tid]; s_cnt[w][tid] = a; a += c; }
  }
  __syncthreads();
  for (int L = 0; L < K; L++) {
    unsigned bal = __ballot_sync(0xffffffffu, (mask >> L) & 1ull);
    if ((mask >> L) & 1ull) {
      int pos = off[L] + tileBase[(long)blockIdx.x * K + L] + s_cnt[wid][L] + __popc(bal & ((1u << lane) - 1u));
      pairs[pos] = pairf(r, L);
    }
  }
}
// write = false: counts and list offsets only (tileCntOut receives the per-tile prefix table for a later k_rule_write)
template <class MaskF, class PairF>
static int build_rule_lists(Metadata &M, int n, int K, MaskF maskf, PairF pairf, RuleBookDev &rb, int extraScalars, bool write = true, int **tileCntOut = nullptr) {
  SCN_CHECK(K >= 1 && K <= 64, "filter volume must be <= 64");
  cudaStream_t s = M.cur().stream;
  rb.nLists = K;
  rb.off.assign(K + 1, 0);
  rb.d_off = M.alloc_n<int>(K + 1);
  int nTiles = cdiv(std::max(n, 1), kRuleTile);
  int *tileCnt = M.alloc_n<int>((long)nTiles * K);
  int *totals = M.cur().d_scalars + 128;
  SCN_CHECK(rb.d_off && tileCnt, "alloc");
  k_rule_count<<<nTiles, kRuleTile, 0, LS(s)>>>(n, K, maskf, tileCnt);
  k_rule_scan<<<K, 1024, 0, LS(s)>>>(nTiles, K, tileCnt, totals);
  k_list_offsets<<<1, 32, 0, LS(s)>>>(K, totals, rb.d_off);
  SCN_CUDA(cudaMemcpyAsync(M.cur().h_scalars + 128, rb.d_off, (K + 1) * 4, cudaMemcpyDeviceToHost, s));
  if (extraScalars) SCN_CUDA(cudaMemcpyAsync(M.cur().h_scalars, M.cur().d_scalars, extraScalars * 4, cudaMemcpyDeviceToHost, s));
  SCN_CUDA(cudaStreamSynchronize(s));
  for (int L = 0; L <= K; L++) rb.off[L] = M.cur().h_scalars[128 + L];
  rb.total = rb.off[K];
  if (tileCntOut) *tileCntOut = tileCnt;
  if (!write) return 0;
  rb.pairs = M.alloc_n<int2>(std::max(1l, rb.total));
  SCN_CHECK(rb.pairs, "alloc");
  if (n > 0) k_rule_write<<<nTiles, kRuleTile, 0, LS(s)>>>(n, K, maskf, pairf, tileCnt, rb.d_off, rb.pairs);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
// More than 64 lists (filter volumes up to kMaxFilterVolume): the same count / scan / write kernels, one pass per 64 lists.  F::word(r, k0)
// gives bits [k0, k0 + 64) of rank r's events; pass w keeps its per-tile prefix table at tileCnt + w nTiles 64.  Each list is
// numbered exactly as above (its position only depends on the earlier ranks with an event in it).
template <class F> struct ChunkMask { F f; int k0; __device__ unsigned long long operator()(int r) const { return f.word(r, k0); } };
template <class F> struct ShiftPair { F f; int k0; __device__ int2 operator()(int r, int L) const { return f(r, L + k0); } };
template <class MaskF, class PairF>
static int write_rule_lists_wide(Metadata &M, int n, int K, MaskF maskf, PairF pairf, const int *tileCnt, const int *d_off, int2 *pairs) {
  const int nTiles = cdiv(std::max(n, 1), kRuleTile);
  for (int k0 = 0; n > 0 && k0 < K; k0 += 64)
    k_rule_write<<<nTiles, kRuleTile, 0, LS(M.cur().stream)>>>(n, std::min(64, K - k0), ChunkMask<MaskF>{maskf, k0}, ShiftPair<PairF>{pairf, k0},
                                                              tileCnt + (long)(k0 / 64) * nTiles * 64, d_off + k0, pairs);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
template <class MaskF, class PairF>
static int build_rule_lists_wide(Metadata &M, int n, int K, MaskF maskf, PairF pairf, RuleBookDev &rb, int extraScalars, bool write = true, int **tileCntOut = nullptr) {
  SCN_CHECK(K > 64 && K <= kMaxFilterVolume, "filter volume must be <= 512");
  cudaStream_t s = M.cur().stream;
  rb.nLists = K;
  rb.off.assign(K + 1, 0);
  rb.d_off = M.alloc_n<int>(K + 1);
  const int nTiles = cdiv(std::max(n, 1), kRuleTile);
  int *tileCnt = M.alloc_n<int>((long)cdiv(K, 64) * nTiles * 64);
  int *totals = M.alloc_n<int>(K);
  SCN_CHECK(rb.d_off && tileCnt && totals, "alloc");
  for (int k0 = 0; k0 < K; k0 += 64) {
    const int Lw = std::min(64, K - k0);
    int *tc = tileCnt + (long)(k0 / 64) * nTiles * 64;
    k_rule_count<<<nTiles, kRuleTile, 0, LS(s)>>>(n, Lw, ChunkMask<MaskF>{maskf, k0}, tc);
    k_rule_scan<<<Lw, 1024, 0, LS(s)>>>(nTiles, Lw, tc, totals + k0);
  }
  k_list_offsets<<<1, 32, 0, LS(s)>>>(K, totals, rb.d_off);
  SCN_CUDA(cudaMemcpyAsync(rb.off.data(), rb.d_off, (K + 1) * 4, cudaMemcpyDeviceToHost, s));
  if (extraScalars) SCN_CUDA(cudaMemcpyAsync(M.cur().h_scalars, M.cur().d_scalars, extraScalars * 4, cudaMemcpyDeviceToHost, s));
  SCN_CUDA(cudaStreamSynchronize(s));
  rb.total = rb.off[K];
  if (tileCntOut) *tileCntOut = tileCnt;
  if (!write) return 0;
  rb.pairs = M.alloc_n<int2>(std::max(1l, rb.total));
  SCN_CHECK(rb.pairs, "alloc");
  return write_rule_lists_wide(M, n, K, maskf, pairf, tileCnt, rb.d_off, rb.pairs);
}

// ------------------------------------------------------------------ per-tile offset masks
__global__ void __launch_bounds__(128) k_tile_masks(const int *__restrict__ nbr, int nOut, int K, unsigned long long *__restrict__ masks) {
  const int tile = blockIdx.x, p = tile * 128 + threadIdx.x;
  unsigned long long m = 0;
  if (p < nOut) {
    for (int k = 0; k < K; k++) m |= (unsigned long long)(nbr[nbr_index(p, k, K)] >= 0) << k;
  }
  for (int d = 16; d > 0; d >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, d);
  __shared__ unsigned long long s[4];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) masks[tile] = s[0] | s[1] | s[2] | s[3];
}
// wide plans: block (tile, chunk) -> the chunk's mask word of the tile (bit j = offset 63 chunk + j), for every tile of the padded plan
__global__ void __launch_bounds__(128) k_tile_masks_wide(const int *__restrict__ nbr, int nOut, int K, long nPad, unsigned long long *__restrict__ masks) {
  const int tile = blockIdx.x, c = blockIdx.y, k0 = c * kChunkOffsets, Kc = min(kChunkOffsets, K - k0);
  const long p = (long)tile * 128 + threadIdx.x;
  unsigned long long m = 0;
  if (p < nOut)
    for (int j = 0; j < Kc; j++) m |= (unsigned long long)(nbr[(long)k0 * nPad + nbr_index(p, j, Kc)] >= 0) << j;
  for (int d = 16; d > 0; d >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, d);
  __shared__ unsigned long long s[4];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) masks[(long)c * (nPad / 128) + tile] = s[0] | s[1] | s[2] | s[3];
}
int Metadata::build_tile_masks(NbrPlan &plan) {
  if (plan.K > 64) {
    const long nPad = plan_padded(plan.nOut);
    plan.tileMask = alloc_n<unsigned long long>(plan_chunks(plan.K) * (nPad / 128) + 8);
    SCN_CHECK(plan.tileMask, "alloc");
    if (plan.nOut > 0)
      k_tile_masks_wide<<<dim3((unsigned)(nPad / 128), plan_chunks(plan.K)), 128, 0, LS(cur().stream)>>>(plan.nbr, plan.nOut, plan.K, nPad, plan.tileMask);
    SCN_CUDA(cudaGetLastError());
    return 0;
  }
  int nTiles = cdiv(std::max(plan.nOut, 1), 128);
  plan.tileMask = alloc_n<unsigned long long>(nTiles + 8);
  SCN_CHECK(plan.tileMask, "alloc");
  if (plan.nOut > 0) k_tile_masks<<<nTiles, 128, 0, LS(cur().stream)>>>(plan.nbr, plan.nOut, plan.K, plan.tileMask);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ submanifold
// nbr[nbr_index(p, k, K)] = row id of the neighbour of site p at filter offset k (last dimension fastest,
// RectangularRegions.h:56-71; window [c - f/2, c + f - 1 - f/2], SubmanifoldConvolutionRules.h:11-22).
// 128 threads per block = one plan tile per loop iteration: the tile's offset mask (bit k: some site of the tile has a
// neighbour at offset k) is reduced on the spot instead of by a second pass over the plan.
//
// SORTED PLANS.  The plan may list the sites in any order (slot q of the plan <-> site perm[q]; outRow[q] names its output row).
// The tensor-core kernel multiplies whole 128-row tiles per live filter offset, so a tile whose sites have DIFFERENT neighbour
// patterns (a piece of floor next to a piece of wall) pays for the union of their offsets with half-empty operand rows: on the
// B470 building 14.9 of 27 offsets are live per tile at a row fill of 62 %.  Inside windows of kSortWindow sites (in spatial
// order, so the gathers stay local) the sites are therefore grouped by the AXES along which they have neighbours (x / y / z: 3
// bits -- floor, the two wall orientations, junctions), stable within a group: 10.4 live offsets per tile, fill 89 %.
constexpr int kSortWindow = 16384;   // sites per window = 128 tiles; one CTA sorts one window
constexpr int kSortMinSites = 4096;  // smaller levels keep the spatial order
__global__ void __launch_bounds__(256) k_site_class(GridView g, const int4 *__restrict__ coords, const int *__restrict__ p2id, int n, int f0, int f1, int f2,
                                                    unsigned char *__restrict__ cls) {
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < n; p += (long)gridDim.x * blockDim.x) {
    const int4 c = coords[p2id[p]];
    int m = 0;
    for (int a = 0; a < f0 && m != 7; a++)
      for (int b = 0; b < f1 && m != 7; b++)
        for (int d = 0; d < f2; d++) {
          const int dx = a - f0 / 2, dy = b - f1 / 2, dz = d - f2 / 2;
          const int bits = (dx ? 4 : 0) | (dy ? 2 : 0) | (dz ? 1 : 0);
          if ((bits & ~m) == 0) continue; // nothing new to learn from this offset (includes the centre)
          if (grid_has(g, c.x + dx, c.y + dy, c.z + dz, c.w)) m |= bits;
        }
    cls[p] = (unsigned char)m;
  }
}
// 3x3x3 filters: the 27-bit neighbour mask of EVERY site of a 64-site occupancy word at once, by shifting occupancy words.
// Bit i of a word = site (y, z) = (i >> 3, i & 7) of one x-slice of an 8x8x8 block; the neighbour at (dy, dz) of all 64 sites is
// the word shifted by 8 dy + dz bits with the bits that cross the block border taken from the adjacent blocks' words.  One thread
// per word: 27 directory / word loads for 64 sites instead of 26 probes (2 loads each) per site.  nmask[p] bit k = filter offset k.
__device__ __forceinline__ unsigned long long shift_z(unsigned long long c, unsigned long long side, int dz) {
  if (dz == 0) return c;
  if (dz > 0) return ((c >> 1) & 0x7f7f7f7f7f7f7f7full) | ((side << 7) & 0x8080808080808080ull);
  return ((c << 1) & 0xfefefefefefefefeull) | ((side >> 7) & 0x0101010101010101ull);
}
__global__ void __launch_bounds__(128) k_word_masks3(GridView g, const int4 *__restrict__ coords, const int *__restrict__ p2id, const int *__restrict__ nblocks,
                                                     unsigned *__restrict__ nmask) {
  const long nWords = (long)(*nblocks) * 8;
  for (long w = blockIdx.x * (long)blockDim.x + threadIdx.x; w < nWords; w += (long)gridDim.x * blockDim.x) {
    const unsigned long long W = g.bmask[w];
    if (!W) continue;
    const int p0 = g.wbase[w];
    const int4 c0 = coords[p2id[p0]]; // any site of the word names its block
    const int bx = c0.x >> 3, by = c0.y >> 3, bz = c0.z >> 3, xs = (int)(w & 7);
    unsigned long long N[27];
#pragma unroll
    for (int a = -1; a <= 1; a++) {
      const int xa = xs + a, bxa = bx + (xa < 0 ? -1 : (xa > 7 ? 1 : 0)), xsa = xa & 7;
      unsigned long long B[3][3]; // occupancy words of x-slice xs + a in the 3 x 3 blocks around (by, bz)
#pragma unroll
      for (int jy = -1; jy <= 1; jy++)
#pragma unroll
        for (int jz = -1; jz <= 1; jz++) {
          const int yy = by + jy, zz = bz + jz;
          unsigned long long v = 0;
          if ((unsigned)bxa < (unsigned)g.dd0 && (unsigned)yy < (unsigned)g.dd1 && (unsigned)zz < (unsigned)g.dd2) {
            const int blk = __ldg(g.dir + (long)c0.w * g.dirCells + ((long)bxa * g.dd1 + yy) * g.dd2 + zz);
            if (blk >= 0) v = __ldg(g.bmask + (long)blk * 8 + xsa);
          }
          B[jy + 1][jz + 1] = v;
        }
#pragma unroll
      for (int dz = -1; dz <= 1; dz++) {
        unsigned long long Z[3];
#pragma unroll
        for (int jy = 0; jy < 3; jy++) Z[jy] = shift_z(B[jy][1], B[jy][1 + (dz == 0 ? 0 : dz)], dz);
#pragma unroll
        for (int dy = -1; dy <= 1; dy++) {
          unsigned long long S = dy == 0 ? Z[1] : (dy > 0 ? ((Z[1] >> 8) | (Z[2] << 56)) : ((Z[1] << 8) | (Z[0] >> 56)));
          N[(a + 1) * 9 + (dy + 1) * 3 + (dz + 1)] = W & S;
        }
      }
    }
    int r = 0;
    for (unsigned long long rest = W; rest; rest &= rest - 1, r++) {
      const int i = __ffsll((long long)rest) - 1;
      unsigned m = 0;
#pragma unroll
      for (int k = 0; k < 27; k++) m |= (unsigned)((N[k] >> i) & 1ull) << k;
      nmask[p0 + r] = m;
    }
  }
}
constexpr unsigned kMaskX = 0x7fc01ffu;  // offsets with dx != 0: k < 9 or k >= 18
constexpr unsigned kMaskY = 0x71f8fc7u;  // dy != 0: (k / 3) % 3 != 1
constexpr unsigned kMaskZ = 0x5b6db6du;  // dz != 0: k % 3 != 1
__global__ void __launch_bounds__(256) k_class_from_mask(const unsigned *__restrict__ nmask, int n, unsigned char *__restrict__ cls) {
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < n; p += (long)gridDim.x * blockDim.x) {
    const unsigned m = nmask[p];
    cls[p] = (unsigned char)(((m & kMaskX) ? 4 : 0) | ((m & kMaskY) ? 2 : 0) | ((m & kMaskZ) ? 1 : 0));
  }
}
// stable counting sort of one window by class: perm[q] = p, slot[p] = q (both in [window start, window end))
__global__ void __launch_bounds__(1024) k_window_sort(const unsigned char *__restrict__ cls, int n, int *__restrict__ perm, int *__restrict__ slot) {
  constexpr int PER = kSortWindow / 1024;
  static_assert(PER == 16, "one 16-byte load per thread");
  __shared__ int s_warp[8][32];
  __shared__ int s_base[8];
  const int w0 = blockIdx.x * kSortWindow, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int p0 = w0 + tid * PER;
  unsigned char mine[PER];
  int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (p0 + PER <= n) { // (cls is 16-byte aligned and padded)
    const uint4 v = *reinterpret_cast<const uint4 *>(cls + p0);
    const unsigned q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < PER; j++) mine[j] = (unsigned char)(q[j >> 2] >> ((j & 3) * 8));
  } else {
#pragma unroll
    for (int j = 0; j < PER; j++) mine[j] = p0 + j < n ? cls[p0 + j] : 255;
  }
#pragma unroll
  for (int j = 0; j < PER; j++) {
#pragma unroll
    for (int c = 0; c < 8; c++) cnt[c] += mine[j] == c;
  }
  int excl[8]; // exclusive prefix of this thread's count within its class, over the threads of the block
#pragma unroll
  for (int c = 0; c < 8; c++) {
    const int inc = warp_incl_scan(cnt[c], lane);
    excl[c] = inc - cnt[c];
    if (lane == 31) s_warp[c][wid] = inc;
  }
  __syncthreads();
  if (wid < 8) { // warp c scans the 32 warp totals of class c
    const int v = s_warp[wid][lane], inc = warp_incl_scan(v, lane);
    s_warp[wid][lane] = inc - v;
    if (lane == 31) s_base[wid] = inc; // class total
  }
  __syncthreads();
  int base = 0;
#pragma unroll
  for (int c = 0; c < 8; c++) {
    excl[c] += s_warp[c][wid] + base;
    base += s_base[c];
  }
#pragma unroll
  for (int j = 0; j < PER; j++) {
    if (p0 + j >= n) break;
    int q = 0;
#pragma unroll
    for (int c = 0; c < 8; c++)
      if (mine[j] == c) q = excl[c]++;
    perm[w0 + q] = p0 + j;
    slot[p0 + j] = w0 + q;
  }
}

__global__ void __launch_bounds__(128) k_subm_nbr(GridView g, const int4 *coords, const int *p2id, int n, int f0, int f1, int f2, int *nbr, int *nValid,
                                                  unsigned long long *tileMask, const int *__restrict__ perm, int *__restrict__ outRow,
                                                  const unsigned *__restrict__ nmask) {
  const int K = f0 * f1 * f2;
  __shared__ unsigned long long s_m[4];
  int cntv = 0;
  const long nPad = ((long)n + 127) / 128 * 128;
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < nPad; p += (long)gridDim.x * blockDim.x) { // p = plan slot
    unsigned long long m = 0;
    if (p < n) {
      const int site = perm ? perm[p] : (int)p; // spatial index of the site in this slot
      const int id = p2id[site];
      if (outRow) outRow[p] = id;
      const int4 c = coords[id];
      const unsigned long long have = nmask ? (unsigned long long)nmask[site] : ~0ull; // known-absent neighbours are not probed
      int k = 0;
      for (int a = 0; a < f0; a++)
        for (int b = 0; b < f1; b++)
          for (int d = 0; d < f2; d++, k++) {
            int x = c.x - f0 / 2 + a, y = c.y - f1 / 2 + b, z = c.z - f2 / 2 + d;
            int q = (x == c.x && y == c.y && z == c.z) ? site : (((have >> k) & 1ull) ? grid_lookup(g, x, y, z, c.w) : -1);
            int v = q >= 0 ? p2id[q] : -1;
            nbr[nbr_index(p, k, K)] = v;
            cntv += v >= 0;
            m |= (unsigned long long)(v >= 0) << k;
          }
    }
    for (int d = 16; d > 0; d >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, d);
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) tileMask[p >> 7] = s_m[0] | s_m[1] | s_m[2] | s_m[3];
    __syncthreads();
  }
  for (int d = 16; d > 0; d >>= 1) cntv += __shfl_xor_sync(0xffffffffu, cntv, d);
  if ((threadIdx.x & 31) == 0 && cntv) atomicAdd(nValid, cntv);
}
// Filters of more than 64 offsets: the same probes into a chunk-major plan (nbr_index_wide); the tile masks are derived from the
// finished plan (k_tile_masks_wide), one word per chunk.
__global__ void __launch_bounds__(128) k_subm_nbr_wide(GridView g, const int4 *coords, const int *p2id, int n, int f0, int f1, int f2, long nPad, int *nbr,
                                                       int *nValid, const int *__restrict__ perm, int *__restrict__ outRow) {
  const int K = f0 * f1 * f2;
  int cntv = 0;
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < n; p += (long)gridDim.x * blockDim.x) { // p = plan slot
    const int site = perm ? perm[p] : (int)p;
    const int id = p2id[site];
    if (outRow) outRow[p] = id;
    const int4 c = coords[id];
    int k = 0;
    for (int a = 0; a < f0; a++)
      for (int b = 0; b < f1; b++)
        for (int d = 0; d < f2; d++, k++) {
          const int x = c.x - f0 / 2 + a, y = c.y - f1 / 2 + b, z = c.z - f2 / 2 + d;
          const int q = (x == c.x && y == c.y && z == c.z) ? site : grid_lookup(g, x, y, z, c.w);
          const int v = q >= 0 ? p2id[q] : -1;
          nbr[nbr_index_wide(p, k, K, nPad)] = v;
          cntv += v >= 0;
        }
  }
  for (int d = 16; d > 0; d >>= 1) cntv += __shfl_xor_sync(0xffffffffu, cntv, d);
  if ((threadIdx.x & 31) == 0 && cntv) atomicAdd(nValid, cntv);
}
struct SubmMaskWide {
  const int *rank2id, *id2p, *nbr; int K; const int *slot; long nPad;
  __device__ unsigned long long word(int r, int k0) const {
    long p = id2p[rank2id[r]];
    if (slot) p = slot[p];
    unsigned long long m = 0;
    for (int k = k0; k < min(K, k0 + 64); k++) m |= (unsigned long long)(nbr[nbr_index_wide(p, k, K, nPad)] >= 0) << (k - k0);
    return m;
  }
};
struct SubmPairWide {
  const int *rank2id, *id2p, *nbr; int K; const int *slot; long nPad;
  __device__ int2 operator()(int r, int L) const {
    int id = rank2id[r];
    long p = id2p[id];
    if (slot) p = slot[p];
    return make_int2(nbr[nbr_index_wide(p, L, K, nPad)], id);
  }
};
struct SubmMask {
  const int *rank2id, *id2p, *nbr; int K; const int *slot;
  __device__ unsigned long long operator()(int r) const {
    long p = id2p[rank2id[r]];
    if (slot) p = slot[p];
    unsigned long long m = 0;
    for (int k = 0; k < K; k++) m |= (unsigned long long)(nbr[nbr_index(p, k, K)] >= 0) << k;
    return m;
  }
};
struct SubmPair {
  const int *rank2id, *id2p, *nbr; int K; const int *slot;
  __device__ int2 operator()(int r, int L) const {
    int id = rank2id[r];
    long p = id2p[id];
    if (slot) p = slot[p];
    return make_int2(nbr[nbr_index(p, L, K)], id); // (input row, output row)
  }
};

// getSubmanifoldRuleBook (Metadata.cpp:429-443) -> SubmanifoldConvolution_SgToRules
// (SubmanifoldConvolutionRules.h:26-45)
int Metadata::get_submanifold(const long *sz, const long *f, SubmEntry **out) {
  SubmKey key{P3{sz[0], sz[1], sz[2]}, P3{f[0], f[1], f[2]}};
  long K = f[0] * f[1] * f[2];
  SCN_CHECK(f[0] > 0 && f[1] > 0 && f[2] > 0 && K <= kMaxFilterVolume, "unsupported submanifold filter size: the filter volume must be <= 512");
  Grid *g = tl_prefetch_worker ? find_grid_wait(sz) : find_grid(sz);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  SubmEntry *ep;
  { std::lock_guard<std::mutex> lk(mapMu); ep = &subm[key]; }
  SubmEntry &e = *ep;
  *out = ep;
  if (!tl_prefetch_worker && !tl_build_here) {
    // The caller shares build context 0 (stream and lock) with the chain worker: a plan the second worker is about
    // to build anyway is waited for instead of being built here, in front of the grid pyramid on the critical path.
    std::unique_lock<std::mutex> lk(mapMu);
    while (e.assigned && !e.rdy.ready && !worker2Done.load()) cv.wait_for(lk, std::chrono::milliseconds(1));
  }
  if (!claim(e.rdy)) return 0; // built (or just finished) by another thread
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, e.rdy};
  BuildLock bl(*this);
  SCN_TRY(need(g->rdy));
  e.plan.K = (int)K;
  e.plan.nOut = g->n;
  e.plan.outRow = g->p2id;
  const long nPad = plan_padded(g->n);
  e.plan.nbr = alloc_n<int>(std::max(1l, nPad * K));
  SCN_CHECK(e.plan.nbr, "alloc");
  const bool wide = K > 64;
  if (wide) { // (every chunk has its own partial last work item)
    SCN_CUDA(cudaMemsetAsync(e.plan.nbr, 0xff, nPad * K * 4, cur().stream));
  } else { // -1 in every slot of the last (partial) work item: whole tiles from the first incomplete one
    const long t0 = (long)g->n / 128;
    SCN_CUDA(cudaMemsetAsync(e.plan.nbr + t0 * K * 128, 0xff, (nPad / 128 - t0) * K * 128 * 4, cur().stream));
  }
  SCN_CUDA(cudaMemsetAsync(cur().d_scalars, 0, 4, cur().stream));
  if (!wide) {
    e.plan.tileMask = alloc_n<unsigned long long>(cdiv(std::max(g->n, 1), 128) + 8);
    SCN_CHECK(e.plan.tileMask, "alloc");
  }
  static int sortOn = -1;
  if (sortOn < 0) sortOn = getenv("SCN_PLAN_SORT") ? atoi(getenv("SCN_PLAN_SORT")) : 1;
  int *perm = nullptr, *outRowSorted = nullptr;
  unsigned *nmask = nullptr;
  if (sortOn && K > 1 && g->n >= kSortMinSites) { // sorted plan (see k_site_class)
    unsigned char *cls = static_cast<unsigned char *>(alloc((size_t)g->n + 16));
    perm = alloc_n<int>(g->n);
    int *slot = alloc_n<int>(g->n);
    outRowSorted = alloc_n<int>(g->n);
    SCN_CHECK(cls && perm && slot && outRowSorted, "alloc");
    if (f[0] == 3 && f[1] == 3 && f[2] == 3) { // neighbour masks of all sites by word shifts; k_subm_nbr then probes present neighbours only
      nmask = alloc_n<unsigned>(g->n);
      SCN_CHECK(nmask, "alloc");
      k_word_masks3<<<stream_grid(g->maxBlocks * 8, 128, 16), 128, 0, LS(cur().stream)>>>(view(*g), g->coords, g->p2id, g->d_nblocks, nmask);
      k_class_from_mask<<<stream_grid(g->n, 256, 8), 256, 0, LS(cur().stream)>>>(nmask, g->n, cls);
    } else
      k_site_class<<<stream_grid(g->n, 256, 8), 256, 0, LS(cur().stream)>>>(view(*g), g->coords, g->p2id, g->n, (int)f[0], (int)f[1], (int)f[2], cls);
    k_window_sort<<<cdiv(g->n, kSortWindow), 1024, 0, LS(cur().stream)>>>(cls, g->n, perm, slot);
    e.plan.outRow = outRowSorted;
    e.plan.slot = slot;
  }
  if (wide) {
    if (g->n) k_subm_nbr_wide<<<stream_grid(g->n, 128, 16), 128, 0, LS(cur().stream)>>>(view(*g), g->coords, g->p2id, g->n, (int)f[0], (int)f[1], (int)f[2], nPad, e.plan.nbr,
                                                                                  cur().d_scalars, perm, outRowSorted);
    SCN_TRY(build_tile_masks(e.plan));
  } else if (g->n) k_subm_nbr<<<stream_grid(g->n, 128, 16), 128, 0, LS(cur().stream)>>>(view(*g), g->coords, g->p2id, g->n, (int)f[0], (int)f[1], (int)f[2], e.plan.nbr, cur().d_scalars, e.plan.tileMask, perm, outRowSorted, nmask);
  // The forward pass only needs the plan and the rule COUNT (the reference's multiply-add counter);
  // the per-offset (in,out) lists in the reference's hash-iteration order are materialised on demand
  // (ensure_subm_rules: backward pass, rulebook inspection).
  SCN_TRY(sync_scalars(1));
  e.plan.nValid = cur().h_scalars[0];
  e.rb.nLists = (int)K;
  e.rb.total = e.plan.nValid;
  e.sz = key.sz;
  SCN_TRY(mark_ready(e.rdy));
  *out = &e;
  return 0;
}
// SubmanifoldConvolution_SgToRules order (SubmanifoldConvolutionRules.h:26-45): sites in hash-iteration order
int Metadata::ensure_subm_rules(SubmEntry &e, bool ahead) {
  if (!claim(e.rulesRdy)) return 0;
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, e.rulesRdy};
  BuildLock bl(*this);
  Grid *g = find_grid(e.sz.data());
  SCN_CHECK(g, "grid");
  SCN_TRY(need(g->rdy));
  SCN_TRY(need(e.rdy));
  SCN_TRY(ensure_rank(*g));
  const int K = e.plan.K;
  if (K > 64) {
    const long nPad = plan_padded(e.plan.nOut);
    SCN_TRY(build_rule_lists_wide(*this, g->n, K, SubmMaskWide{g->rank2id, g->id2p, e.plan.nbr, K, e.plan.slot, nPad},
                                  SubmPairWide{g->rank2id, g->id2p, e.plan.nbr, K, e.plan.slot, nPad}, e.rb, 0));
  } else {
    SCN_TRY(build_rule_lists(*this, g->n, K, SubmMask{g->rank2id, g->id2p, e.plan.nbr, K, e.plan.slot}, SubmPair{g->rank2id, g->id2p, e.plan.nbr, K, e.plan.slot}, e.rb, 0));
  }
  SCN_CHECK(e.plan.nValid == e.rb.total, "internal: rule count mismatch");
  e.rulesRdy.ahead = ahead;
  return mark_ready(e.rulesRdy);
}

// ------------------------------------------------------------------ strided convolution
typedef ConvGeomHost ConvGeom;
// output cells of input point c: [lb, ub] per dim (OutputRegionCalculator, RectangularRegions.h:109-119);
// event m enumerates them last-dimension-fastest.  Returns false when m is outside the region.
__device__ __forceinline__ bool conv_event(const ConvGeom &G, const int4 &c, int m, int4 &j, int &off) {
  int a[3];
  a[2] = m % G.cnt[2]; m /= G.cnt[2];
  a[1] = m % G.cnt[1]; m /= G.cnt[1];
  a[0] = m;
  const int p[3] = {c.x, c.y, c.z};
  int jj[3];
  off = 0;
  for (int d = 0; d < 3; d++) {
    int lo = (p[d] - G.f[d] + G.s[d]) / G.s[d]; // C++ truncating division, as the reference
    if (lo < 0) lo = 0;
    int hi = min(G.outS[d] - 1, p[d] / G.s[d]);
    jj[d] = lo + a[d];
    if (jj[d] > hi) return false;
    off = off * G.f[d] + (p[d] - jj[d] * G.s[d]); // RectangularRegion::offset, :30-38
  }
  j = make_int4(jj[0], jj[1], jj[2], c.w);
  return true;
}
__global__ void k_conv_events(ConvGeom G, const int *rank2id, const int4 *coords, int n, int4 *evPts) {
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < (long)n * G.M; e += (long)gridDim.x * blockDim.x) {
    int r = (int)(e / G.M), m = (int)(e % G.M);
    int4 c = coords[rank2id[r]], j;
    int off;
    evPts[e] = conv_event(G, c, m, j, off) ? j : make_int4(-1, 0, 0, 0);
  }
}
__global__ void k_first_event(const int *evQ, long E, int *firstEv) {
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < E; e += (long)gridDim.x * blockDim.x) {
    int q = evQ[e];
    if (q >= 0) atomicMin(firstEv + q, (int)e);
  }
}
struct EvFirstIn {
  const int *evQ, *firstEv;
  __device__ int operator()(long e) const { int q = evQ[e]; return q >= 0 && firstEv[q] == (int)e; }
};
struct EvFirstOut {
  const int *evQ; const int4 *evPts; int *p2id, *id2p; int4 *coords; int *batchCnt;
  __device__ void operator()(long e, int pre, int v) const {
    // per-item counts only when there is more than one batch item: with one item every output site would
    // hit the same counter (283K serialised atomics = 0.2 ms at level 0 -> 1 of B470); the caller uses nOut then
    if (v) { int q = evQ[e]; p2id[q] = pre; id2p[pre] = q; coords[pre] = evPts[e]; if (batchCnt) atomicAdd(batchCnt + evPts[e].w, 1); }
  }
};
struct ConvMask {
  ConvGeom G; const int *rank2id; const int4 *coords;
  __device__ unsigned long long operator()(int r) const {
    int4 c = coords[rank2id[r]], j;
    unsigned long long m = 0;
    for (int e = 0; e < G.M; e++) { int off; if (conv_event(G, c, e, j, off)) m |= 1ull << off; }
    return m;
  }
  __device__ unsigned long long word(int r, int k0) const { // filters of more than 64 offsets: offsets [k0, k0 + 64)
    int4 c = coords[rank2id[r]], j;
    unsigned long long m = 0;
    for (int e = 0; e < G.M; e++) { int off; if (conv_event(G, c, e, j, off) && (unsigned)(off - k0) < 64u) m |= 1ull << (off - k0); }
    return m;
  }
};
struct ConvPair {
  ConvGeom G; const int *rank2id; const int4 *coords; const int *evQ; const int *outP2id;
  __device__ int2 operator()(int r, int L) const {
    int id = rank2id[r];
    int4 c = coords[id], j;
    for (int e = 0; e < G.M; e++) { int off; if (conv_event(G, c, e, j, off) && off == L) return make_int2(id, outP2id[evQ[(long)r * G.M + e]]); }
    return make_int2(-1, -1);
  }
};
__global__ void k_conv_plan(ConvGeom G, const int *rank2id, const int4 *coords, const int *evQ, int n, int *nbr) {
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < (long)n * G.M; e += (long)gridDim.x * blockDim.x) {
    int q = evQ[e];
    if (q < 0) continue;
    int r = (int)(e / G.M), m = (int)(e % G.M);
    int id = rank2id[r];
    int4 j; int off;
    conv_event(G, coords[id], m, j, off);
    nbr[nbr_index(q, off, G.K)] = id;
  }
}
__global__ void k_conv_plan_wide(ConvGeom G, const int *rank2id, const int4 *coords, const int *evQ, int n, long nPad, int *nbr) {
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < (long)n * G.M; e += (long)gridDim.x * blockDim.x) {
    int q = evQ[e];
    if (q < 0) continue;
    int r = (int)(e / G.M), m = (int)(e % G.M);
    int id = rank2id[r];
    int4 j; int off;
    conv_event(G, coords[id], m, j, off);
    nbr[nbr_index_wide(q, off, G.K, nPad)] = id;
  }
}

// ------------------------------------------------------------------ small levels: one launch per strided convolution
// The deep pyramid levels hold a few thousand sites, yet the general path above spends ~25 launches and 3 host
// round trips on each (measured: ~0.3 ms per level, all of it launch latency, and the grid pyramid is the critical
// path of the forward).  For an input grid of <= kSmallSites sites (one batch item, one output cell per site) ONE CTA
// does the whole build -- hash-iteration order, output grid, first-touch numbering, rule lists in reference order,
// execution plan, tile masks -- with __syncthreads between the steps, and the host reads the counts back once.
// Same algorithm, same results as the multi-launch path (tests compare both against the reference rulebooks).
constexpr int kSmallSites = kSmallNb / 2;
struct ConvSmallArgs {
  const int4 *inCoords; int n, idOffset, doRank, spatial; int *rank2id;
  ConvGeom G;
  int *dir; unsigned long long *bmask; int *wbase; int *d_nblocks; int cells, dd1, dd2; int sz0, sz1, sz2; int cap;
  int4 *evPts; int *evQ, *evOff, *firstEv;
  int4 *oCoords; int *p2id, *id2p;
  int2 *pairs; int *d_off;
  int *nbr; unsigned long long *tileMask; int nTilesCap;
  int *sc, *err;
};
// exclusive scan over n items by the whole CTA (1024 threads, item i handled by thread i % 1024); returns the total
template <class InF, class OutF>
__device__ __forceinline__ int cta_scan(int n, InF in, OutF out, int *s_scan /* [33] */) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int carry = 0;
  for (int base = 0; base < n; base += 1024) {
    const int i = base + tid;
    const int v = i < n ? in(i) : 0;
    const int incl = warp_incl_scan(v, lane);
    if (lane == 31) s_scan[wid] = incl;
    __syncthreads();
    if (wid == 0) { int w = s_scan[lane]; int wi = warp_incl_scan(w, lane); s_scan[lane] = wi - w; if (lane == 31) s_scan[32] = wi; }
    __syncthreads();
    if (i < n) out(i, carry + s_scan[wid] + incl - v, v);
    carry += s_scan[32];
    __syncthreads();
  }
  return carry;
}
__global__ void __launch_bounds__(1024) k_conv_small(const ConvSmallArgs A) {
  extern __shared__ unsigned sm[];
  __shared__ int s_scan[33];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = A.n, K = A.G.K;
  // ---- reference hash-iteration order of the input grid
  if (A.doRank && A.spatial) {
    for (int r = tid; r < n; r += 1024) A.rank2id[r] = r + A.idOffset;
  } else if (A.doRank) {
    const SmallEmu e = emulate_small_body(A.inCoords, nullptr, A.idOffset, n, sm, A.cap, A.err);
    cta_scan(e.nb, [&](int i) { return e.tab[i] != kEmpty; },
             [&](int i, int pre, int v) { if (v) A.rank2id[pre] = e.seq[e.tab[i] >> kProbeBits]; }, s_scan);
  }
  __syncthreads();
  // ---- events (one per input site, rank order) and the block directory of the output grid
  for (int r = tid; r < n; r += 1024) {
    const int4 c = A.inCoords[__ldcg(A.rank2id + r)];
    int4 j; int off;
    bool ok = conv_event(A.G, c, 0, j, off);
    if (ok && (j.x >= A.sz0 || (unsigned)j.y >= (unsigned)A.sz1 || (unsigned)j.z >= (unsigned)A.sz2)) { *A.err = 2; ok = false; }
    A.evPts[r] = ok ? j : make_int4(-1, 0, 0, 0);
    A.evOff[r] = ok ? off : -1;
    if (ok) A.dir[((j.x >> 3) * A.dd1 + (j.y >> 3)) * A.dd2 + (j.z >> 3)] = 1;
  }
  __syncthreads();
  const int nblocks = cta_scan(A.cells, [&](int i) { return __ldcg(A.dir + i) != 0; }, [&](int i, int pre, int v) { A.dir[i] = v ? pre : -1; }, s_scan);
  if (tid == 0) *A.d_nblocks = nblocks;
  for (int i = tid; i < nblocks * 8; i += 1024) A.bmask[i] = 0ull;
  __syncthreads();
  for (int r = tid; r < n; r += 1024) {
    if (A.evOff[r] < 0) continue;
    const int4 j = A.evPts[r];
    const int blk = __ldcg(A.dir + ((j.x >> 3) * A.dd1 + (j.y >> 3)) * A.dd2 + (j.z >> 3));
    const int bit = ((j.x & 7) << 6) | ((j.y & 7) << 3) | (j.z & 7);
    atomicOr(A.bmask + (long)blk * 8 + (bit >> 6), 1ull << (bit & 63));
  }
  __syncthreads();
  const int nunique = cta_scan(nblocks * 8, [&](int i) { return __popcll(__ldcg(A.bmask + i)); }, [&](int i, int pre, int) { A.wbase[i] = pre; }, s_scan);
  // ---- spatial index of every event, first event per output site
  for (int r = tid; r < n; r += 1024) {
    int q = -1;
    if (A.evOff[r] >= 0) {
      const int4 j = A.evPts[r];
      const int blk = __ldcg(A.dir + ((j.x >> 3) * A.dd1 + (j.y >> 3)) * A.dd2 + (j.z >> 3));
      const int bit = ((j.x & 7) << 6) | ((j.y & 7) << 3) | (j.z & 7);
      const int w = blk * 8 + (bit >> 6);
      const unsigned long long m = __ldcg(A.bmask + w), one = 1ull << (bit & 63);
      q = __ldcg(A.wbase + w) + __popcll(m & (one - 1));
      atomicMin(A.firstEv + q, r);
    }
    A.evQ[r] = q;
  }
  __syncthreads();
  // ---- first-touch numbering of the output sites (ConvolutionRules.h:19-31)
  int nOut;
  if (A.spatial) { // row id = spatial index
    for (int r = tid; r < n; r += 1024) {
      const int q = A.evQ[r];
      if (q >= 0 && __ldcg(A.firstEv + q) == r) { A.p2id[q] = q; A.id2p[q] = q; A.oCoords[q] = A.evPts[r]; }
    }
    nOut = nunique;
    __syncthreads();
  } else {
    nOut = cta_scan(n, [&](int r) { const int q = A.evQ[r]; return (int)(q >= 0 && __ldcg(A.firstEv + q) == r); },
                    [&](int r, int pre, int v) { if (v) { const int q = A.evQ[r]; A.p2id[q] = pre; A.id2p[pre] = q; A.oCoords[pre] = A.evPts[r]; } }, s_scan);
  }
  // ---- rule lists: list L holds the (input row, output row) pairs of the events with offset L, in rank order
  int *s_tot = reinterpret_cast<int *>(sm), *s_off = s_tot + 64;
  int(*s_w)[64] = reinterpret_cast<int(*)[64]>(sm + 192);
  if (tid < 64) s_tot[tid] = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int r = base + tid, L = r < n ? A.evOff[r] : -1;
    for (int l = 0; l < K; l++) {
      const unsigned bal = __ballot_sync(0xffffffffu, L == l);
      if (lane == 0 && bal) atomicAdd(s_tot + l, __popc(bal));
    }
  }
  __syncthreads();
  if (tid == 0) {
    int a = 0;
    for (int l = 0; l < K; l++) { s_off[l] = a; A.d_off[l] = a; A.sc[128 + l] = a; a += s_tot[l]; }
    s_off[K] = a; A.d_off[K] = a; A.sc[128 + K] = a;
    A.sc[1] = nunique; A.sc[3] = nOut;
  }
  __syncthreads();
  if (tid < 64) s_tot[tid] = 0; // from here: pairs already written per list
  for (int t = tid; t < A.nTilesCap; t += 1024) A.tileMask[t] = 0ull;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int r = base + tid, L = r < n ? A.evOff[r] : -1;
    unsigned mine = 0;
    for (int l = 0; l < K; l++) {
      const unsigned bal = __ballot_sync(0xffffffffu, L == l);
      if (lane == 0) s_w[wid][l] = __popc(bal);
      if (L == l) mine = bal;
    }
    __syncthreads();
    if (tid < K) {
      int a = s_tot[tid];
      for (int w = 0; w < 32; w++) { const int c = s_w[w][tid]; s_w[w][tid] = a; a += c; }
      s_tot[tid] = a;
    }
    __syncthreads();
    if (L >= 0) {
      const int id = __ldcg(A.rank2id + r), q = A.evQ[r];
      A.pairs[s_off[L] + s_w[wid][L] + __popc(mine & ((1u << lane) - 1u))] = make_int2(id, __ldcg(A.p2id + q));
      // output-stationary plan + per-tile offset masks
      A.nbr[nbr_index(q, L, K)] = id;
      atomicOr(A.tileMask + (q >> 7), 1ull << L);
    }
    __syncthreads();
  }
}
int Metadata::get_conv_small(Grid &gi, Grid &go, ConvEntry &e, const ConvGeomHost &G) {
  cudaStream_t s = cur().stream;
  const int n = gi.n;
  const bool doRank = claim(gi.rankRdy);
  struct Guard { Metadata &m; Ready &r; bool on; ~Guard() { if (on && !r.ready) m.unclaim(r); } } guard{*this, gi.rankRdy, doRank};
  if (doRank) { gi.rank2id = alloc_n<int>(n); SCN_CHECK(gi.rank2id, "alloc"); }
  else SCN_TRY(need(gi.rankRdy));
  for (int d = 0; d < 3; d++) go.dd[d] = (int)((go.sz[d] + 7) / 8);
  go.dirCells = (long)go.dd[0] * go.dd[1] * go.dd[2];
  const long cells = go.dirCells;
  go.dir = alloc_n<int>(cells);
  go.d_nblocks = alloc_n<int>(4);
  go.maxBlocks = std::max(1l, std::min<long>(n, cells));
  go.bmask = alloc_n<unsigned long long>(go.maxBlocks * 8);
  go.wbase = alloc_n<int>(go.maxBlocks * 8);
  go.coords = alloc_n<int4>(n); go.p2id = alloc_n<int>(n); go.id2p = alloc_n<int>(n);
  int4 *evPts = alloc_n<int4>(n);
  int *evQ = alloc_n<int>(n), *evOff = alloc_n<int>(n), *firstEv = alloc_n<int>(n);
  const long nPad = plan_padded(n);
  const int nTilesCap = (int)(nPad / 128);
  e.rb.nLists = G.K;
  e.rb.d_off = alloc_n<int>(G.K + 1);
  e.rb.pairs = alloc_n<int2>(n);
  e.plan.nbr = alloc_n<int>(nPad * G.K);
  e.plan.tileMask = alloc_n<unsigned long long>(nTilesCap + 8);
  SCN_CHECK(go.dir && go.d_nblocks && go.bmask && go.wbase && go.coords && go.p2id && go.id2p && evPts && evQ && evOff && firstEv && e.rb.d_off &&
                e.rb.pairs && e.plan.nbr && e.plan.tileMask, "alloc");
  int *sc = cur().d_scalars;
  SCN_CUDA(cudaMemsetAsync(go.dir, 0, cells * 4, s));
  SCN_CUDA(cudaMemsetAsync(firstEv, 0x7f, (size_t)n * 4, s));
  SCN_CUDA(cudaMemsetAsync(e.plan.nbr, 0xff, (size_t)nPad * G.K * 4, s));
  ConvSmallArgs A;
  A.inCoords = gi.coords; A.n = n; A.idOffset = gi.itemCtr[0]; A.doRank = doRank ? 1 : 0; A.spatial = spatialIds ? 1 : 0; A.rank2id = gi.rank2id;
  A.G = G;
  A.dir = go.dir; A.bmask = go.bmask; A.wbase = go.wbase; A.d_nblocks = go.d_nblocks; A.cells = (int)cells; A.dd1 = go.dd[1]; A.dd2 = go.dd[2];
  A.sz0 = (int)go.sz[0]; A.sz1 = (int)go.sz[1]; A.sz2 = (int)go.sz[2];
  A.evPts = evPts; A.evQ = evQ; A.evOff = evOff; A.firstEv = firstEv;
  A.oCoords = go.coords; A.p2id = go.p2id; A.id2p = go.id2p;
  A.pairs = e.rb.pairs; A.d_off = e.rb.d_off;
  A.nbr = e.plan.nbr; A.tileMask = e.plan.tileMask; A.nTilesCap = nTilesCap;
  A.sc = sc; A.err = cur().d_err;
  int capB = 32;
  while (n > capB / 2) capB *= 2; // final table of the hash-order emulation (n <= kSmallSites => capB <= kSmallNb)
  A.cap = capB;
  const int smem = std::max(3 * capB * 4, 10 * 1024); // the rule-list pass reuses the buffer (9 KB)
  static bool attr = false;
  if (!attr) { SCN_CUDA(cudaFuncSetAttribute(k_conv_small, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * kSmallNb * 4)); attr = true; }
  k_conv_small<<<1, 1024, smem, LS(s)>>>(A);
  SCN_CUDA(cudaGetLastError());
  SCN_CUDA(cudaMemcpyAsync(cur().h_scalars, sc, (128 + G.K + 1) * 4, cudaMemcpyDeviceToHost, s));
  SCN_CUDA(cudaStreamSynchronize(s));
  if (doRank) { gi.hasRank = true; SCN_TRY(mark_ready(gi.rankRdy)); }
  e.rb.off.assign(G.K + 1, 0);
  for (int L = 0; L <= G.K; L++) e.rb.off[L] = cur().h_scalars[128 + L];
  e.rb.total = e.rb.off[G.K];
  go.n = cur().h_scalars[3];
  SCN_CHECK(cur().h_scalars[1] == go.n, "internal: unique count mismatch (small conv)");
  go.itemCount.assign(1, go.n);
  go.itemCtr.assign(1, 0);
  e.plan.K = G.K; e.plan.nOut = go.n; e.plan.outRow = go.p2id; e.plan.nValid = e.rb.total;
  return 0;
}

static int conv_geom(const long *f, const long *st, const long *outS, ConvGeom &G) {
  G.M = 1; G.K = 1;
  for (int d = 0; d < 3; d++) {
    SCN_CHECK(f[d] >= 1 && st[d] >= 1 && outS[d] >= 1, "bad filter geometry");
    G.f[d] = (int)f[d]; G.s[d] = (int)st[d]; G.outS[d] = (int)outS[d];
    G.cnt[d] = (int)std::min<long>(outS[d], (f[d] + st[d] - 1) / st[d]);
    if (G.cnt[d] < 1) G.cnt[d] = 1;
    G.M *= G.cnt[d]; G.K *= (int)f[d];
  }
  SCN_CHECK(G.K <= kMaxFilterVolume && G.M <= 64, "unsupported convolution filter size: the filter volume must be <= 512 and the output cells per input site <= 64");
  return 0;
}
// get_conv_small serves this convolution (one launch builds the output grid, its numbering, the lists and the plan)
static bool small_conv(const Grid &gi, const ConvGeom &G, const long *outS) {
  static int smallOn = -1;
  if (smallOn < 0) smallOn = getenv("SCN_SMALL_FUSED") ? atoi(getenv("SCN_SMALL_FUSED")) : 1;
  return smallOn && G.M == 1 && G.K <= 64 && gi.batch == 1 && gi.n > 0 && gi.n <= kSmallSites && gi.itemCtr.size() == 1 && gi.itemCtr[0] >= 0 &&
         ((outS[0] + 7) / 8) * ((outS[1] + 7) / 8) * ((outS[2] + 7) / 8) <= (1 << 16);
}

// getRuleBook (Metadata.cpp:484-510) -> Convolution_InputSgToRulesAndOutputSg (ConvolutionRules.h:11-34)
int Metadata::get_conv(const long *inS, const long *outS, const long *f, const long *st, ConvEntry **out) {
  ConvKey key{P3{inS[0], inS[1], inS[2]}, P3{f[0], f[1], f[2]}, P3{st[0], st[1], st[2]}};
  Grid *gi = tl_prefetch_worker ? find_grid_wait(inS) : find_grid(inS);
  SCN_CHECK(gi, "no active sites recorded for the input spatial size");
  P3 okey{outS[0], outS[1], outS[2]};
  ConvEntry *ep;
  { std::lock_guard<std::mutex> lk(mapMu); ep = &conv[key]; }
  *out = ep;
  if (!claim(ep->rdy)) return 0; // built (or just finished) by another thread
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, ep->rdy};
  BuildLock bl(*this);
  SCN_TRY(need(gi->rdy));
  ConvEntry &e = *ep;
  // gridGiven: overlay_conv made the output grid (numbering included) and the events' spatial indices evQ; what is left are the
  // rule counts, the plan and the tile masks over that grid
  const bool given = e.gridGiven;
  {
    std::lock_guard<std::mutex> lk(mapMu);
    SCN_CHECK(given ? e.out == okey : grids.find(okey) == grids.end(), "output spatial size already has a grid (each spatial size may occur once per Metadata)");
  }
  ConvGeom G;
  SCN_TRY(conv_geom(f, st, outS, G));
  Grid *gop;
  { std::lock_guard<std::mutex> lk(mapMu); gop = &grids[okey]; }
  e.out = okey;
  e.in = key.in;
  e.geom = G;
  Grid &go = *gop;
  if (!given && small_conv(*gi, G, outS)) {
    go.sz = okey;
    go.batch = gi->batch;
    SCN_TRY(get_conv_small(*gi, go, e, G));
    SCN_TRY(mark_ready(e.rulesRdy)); // the one-launch build writes the lists as well
    SCN_TRY(mark_ready(go.rdy));
    { std::lock_guard<std::mutex> lk(mapMu); go.built = true; }
    cv.notify_all();
    SCN_TRY(mark_ready(e.rdy));
    return 0;
  }
  SCN_TRY(ensure_rank(*gi));
  cudaStream_t s = cur().stream;
  const int n = gi->n;
  const long E = (long)n * G.M;
  const int *evQ = e.evQ;
  if (given) SCN_TRY(need(go.rdy));
  else {
    go.sz = okey;
    go.batch = gi->batch;
    int4 *evPts = alloc_n<int4>(std::max(1l, E));
    int *q = alloc_n<int>(std::max(1l, E));
    SCN_CHECK(evPts && q, "alloc");
    int *sc = cur().d_scalars; // [1] nunique [3] nOut [8..56) per-item counts
    SCN_CUDA(cudaMemsetAsync(sc, 0, 64 * 4, s));
    if (E) k_conv_events<<<stream_grid(E, 256), 256, 0, LS(s)>>>(G, gi->rank2id, gi->coords, n, evPts);
    SCN_TRY(build_blocks(*this, go, evPts, E, q, sc + 1));
    long cap = std::max(1l, E);
    go.coords = alloc_n<int4>(cap); go.p2id = alloc_n<int>(cap); go.id2p = alloc_n<int>(cap);
    int *firstEv = alloc_n<int>(cap);
    SCN_CHECK(go.coords && go.p2id && go.id2p && firstEv, "alloc");
    if (spatialIds) {
      if (E) k_spatial_conv_ids<<<stream_grid(E, 256), 256, 0, LS(s)>>>(q, evPts, E, go.coords, go.p2id, go.id2p);
      k_copy_scalar<<<1, 1, 0, LS(s)>>>(sc + 1, sc + 3);
    } else {
      SCN_CUDA(cudaMemsetAsync(firstEv, 0x7f, cap * 4, s));
      if (E) k_first_event<<<stream_grid(E, 256), 256, 0, LS(s)>>>(q, E, firstEv);
      SCN_TRY(run_scan(*this, E, EvFirstIn{q, firstEv}, EvFirstOut{q, evPts, go.p2id, go.id2p, go.coords, go.batch > 1 ? sc + 8 : nullptr}, sc + 3));
    }
    evQ = q;
  }
  // rule lists (one sync: list offsets + nOut + per-item counts)
  const int extra = given ? 0 : 64;
  if (G.K > 64)
    SCN_TRY(build_rule_lists_wide(*this, n, G.K, ConvMask{G, gi->rank2id, gi->coords},
                                  ConvPair{G, gi->rank2id, gi->coords, evQ, go.p2id}, e.rb, extra, /*write=*/false, &e.tileCnt));
  else
    SCN_TRY(build_rule_lists(*this, n, G.K, ConvMask{G, gi->rank2id, gi->coords},
                             ConvPair{G, gi->rank2id, gi->coords, evQ, go.p2id}, e.rb, extra, /*write=*/false, &e.tileCnt));
  e.evQ = evQ;
  if (!given) {
    go.n = cur().h_scalars[3];
    SCN_CHECK(cur().h_scalars[1] == go.n, "internal: unique count mismatch (conv)");
    go.itemCount.assign(go.batch, 0);
    go.itemCtr.assign(go.batch, 0);
    int ctr = 0;
    for (int b = 0; b < go.batch; b++) { go.itemCount[b] = go.batch > 1 ? cur().h_scalars[8 + b] : go.n; go.itemCtr[b] = ctr; ctr += go.itemCount[b]; }
  }
  // output-stationary plan
  e.plan.K = G.K; e.plan.nOut = go.n; e.plan.outRow = go.p2id; e.plan.nValid = e.rb.total;
  const long nPadOut = plan_padded(go.n);
  e.plan.nbr = alloc_n<int>(std::max(1l, nPadOut * G.K));
  SCN_CHECK(e.plan.nbr, "alloc");
  SCN_CUDA(cudaMemsetAsync(e.plan.nbr, 0xff, std::max(1l, nPadOut * G.K) * 4, s));
  if (E && G.K > 64) k_conv_plan_wide<<<stream_grid(E, 256), 256, 0, LS(s)>>>(G, gi->rank2id, gi->coords, evQ, n, nPadOut, e.plan.nbr);
  else if (E) k_conv_plan<<<stream_grid(E, 256), 256, 0, LS(s)>>>(G, gi->rank2id, gi->coords, evQ, n, e.plan.nbr);
  SCN_CUDA(cudaGetLastError());
  SCN_TRY(build_tile_masks(e.plan));
  if (!given) {
    SCN_TRY(mark_ready(go.rdy)); // the event first: a thread that sees `built` must also see the event to wait for
    { std::lock_guard<std::mutex> lk(mapMu); go.built = true; }
    cv.notify_all();
  }
  SCN_TRY(mark_ready(e.rdy));
  return 0;
}

// Output level of a strided convolution, numbered as get_conv numbers it: the events of the input sites in hash-iteration order
// find their spatial index in the internal output grid (whose block structure this grid copies) and the first-touch scan turns
// them into reference ids.  Rule lists and plan are left to get_conv (entry.gridGiven), which nothing in a replayed forward
// calls.  Small levels take the one-launch get_conv as they are.
int Metadata::overlay_conv(Metadata &in, const long *inS, const long *outS, const long *f, const long *st) {
  Grid *gi = find_grid(inS);
  SCN_CHECK(gi, "numbering overlay: no grid of the input spatial size");
  ConvGeom G;
  SCN_TRY(conv_geom(f, st, outS, G));
  if (small_conv(*gi, G, outS)) {
    ConvEntry *e;
    return get_conv(inS, outS, f, st, &e);
  }
  SCN_CHECK(gi->batch == 1, "numbering overlay: one batch item");
  BuildLock bl(*this);
  SCN_TRY(need(gi->rdy));
  SCN_TRY(ensure_rank(*gi)); // first: the hash-order emulation does not need the internal output grid
  Grid *gq = internal_grid(*this, in, outS);
  if (!gq) { // not made by `in`'s chain worker (a leaf of the pyramid, built later by another thread): the complete build
    ConvEntry *e;
    return get_conv(inS, outS, f, st, &e);
  }
  ConvEntry *ep;
  {
    std::lock_guard<std::mutex> lk(mapMu);
    ep = &conv[ConvKey{P3{inS[0], inS[1], inS[2]}, P3{f[0], f[1], f[2]}, P3{st[0], st[1], st[2]}}];
  }
  SCN_CHECK(!ep->rdy.ready && !ep->rdy.building && !ep->gridGiven, "numbering overlay: convolution already built");
  Grid *gop = new_grid(*this, outS);
  SCN_CHECK(gop, "output spatial size already has a grid (each spatial size may occur once per Metadata)");
  Grid &go = *gop;
  cudaStream_t s = cur().stream;
  go.batch = 1;
  go.n = gq->n;
  SCN_TRY(copy_blocks(*this, go, *gq));
  const int n = gi->n;
  const long E = (long)n * G.M, cap = std::max(1, go.n);
  int4 *evPts = alloc_n<int4>(std::max(1l, E));
  int *evQ = alloc_n<int>(std::max(1l, E)), *firstEv = alloc_n<int>(cap);
  go.coords = alloc_n<int4>(cap); go.p2id = alloc_n<int>(cap); go.id2p = alloc_n<int>(cap);
  SCN_CHECK(evPts && evQ && firstEv && go.coords && go.p2id && go.id2p, "alloc");
  SCN_CUDA(cudaMemsetAsync(firstEv, 0x7f, cap * 4, s));
  if (E) {
    k_conv_events<<<stream_grid(E, 256), 256, 0, LS(s)>>>(G, gi->rank2id, gi->coords, n, evPts);
    k_lookup_pts<<<stream_grid(E, 256), 256, 0, LS(s)>>>(view(go), evPts, E, evQ);
    k_first_event<<<stream_grid(E, 256), 256, 0, LS(s)>>>(evQ, E, firstEv);
  }
  SCN_TRY(run_scan(*this, E, EvFirstIn{evQ, firstEv}, EvFirstOut{evQ, evPts, go.p2id, go.id2p, go.coords, nullptr}, nullptr));
  {
    std::lock_guard<std::mutex> lk(mapMu);
    ep->in = P3{inS[0], inS[1], inS[2]};
    ep->out = go.sz;
    ep->geom = G;
    ep->evQ = evQ;
    ep->gridGiven = true;
  }
  return publish_grid(*this, go);
}

// The (in,out) lists of a strided convolution in the reference's order (ConvolutionRules.h:11-34), written on demand.
int Metadata::ensure_conv_rules(ConvEntry &e, bool ahead) {
  if (!claim(e.rulesRdy)) return 0;
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, e.rulesRdy};
  BuildLock bl(*this);
  Grid *gi = find_grid(e.in.data()), *go = find_grid(e.out.data());
  SCN_CHECK(gi && go && e.evQ && e.tileCnt, "convolution rulebook not built");
  SCN_TRY(need(e.rdy));
  SCN_TRY(need(gi->rankRdy));
  const int n = gi->n, K = e.geom.K;
  e.rb.pairs = alloc_n<int2>(std::max(1l, e.rb.total));
  SCN_CHECK(e.rb.pairs, "alloc");
  if (K > 64)
    SCN_TRY(write_rule_lists_wide(*this, n, K, ConvMask{e.geom, gi->rank2id, gi->coords}, ConvPair{e.geom, gi->rank2id, gi->coords, e.evQ, go->p2id},
                                  e.tileCnt, e.rb.d_off, e.rb.pairs));
  else if (n > 0)
    k_rule_write<<<cdiv(n, kRuleTile), kRuleTile, 0, LS(cur().stream)>>>(n, K, ConvMask{e.geom, gi->rank2id, gi->coords},
                                                                         ConvPair{e.geom, gi->rank2id, gi->coords, e.evQ, go->p2id}, e.tileCnt, e.rb.d_off, e.rb.pairs);
  SCN_CUDA(cudaGetLastError());
  e.rulesRdy.ahead = ahead;
  return mark_ready(e.rulesRdy);
}

// ------------------------------------------------------------------ deconvolution plan
struct DeconvMask {
  ConvGeom G; const int *p2id; const int4 *coords;
  __device__ unsigned long long operator()(int p) const {
    int4 j; int off;
    return conv_event(G, coords[p2id[p]], 0, j, off) ? 1ull << off : 0ull;
  }
  __device__ unsigned long long word(int p, int k0) const {
    int4 j; int off;
    return conv_event(G, coords[p2id[p]], 0, j, off) && (unsigned)(off - k0) < 64u ? 1ull << (off - k0) : 0ull;
  }
};
struct DeconvPair {
  ConvGeom G; const int *p2id; const int4 *coords; GridView coarse; const int *coarseP2id;
  __device__ int2 operator()(int p, int) const {
    int id = p2id[p];
    int4 j; int off;
    conv_event(G, coords[id], 0, j, off);
    int q = grid_lookup(coarse, j.x, j.y, j.z, j.w);
    return make_int2(q >= 0 ? coarseP2id[q] : -1, id); // (coarse source row, fine destination row)
  }
};
__global__ void k_deconv_pad(const int2 *__restrict__ pairs, const int *__restrict__ off, const int *__restrict__ tileW, const int *__restrict__ tileFirst,
                             int nTiles, int *__restrict__ nbr, int *__restrict__ outRow, unsigned long long *__restrict__ tileMask) {
  for (long slot = blockIdx.x * (long)blockDim.x + threadIdx.x; slot < (long)nTiles * 128; slot += (long)gridDim.x * blockDim.x) {
    int tile = (int)(slot >> 7), k = tileW[tile];
    int idx = (tile - tileFirst[k]) * 128 + (int)(slot & 127);
    int2 pr = make_int2(-1, -1);
    if (idx < off[k + 1] - off[k]) pr = pairs[off[k] + idx];
    nbr[slot] = pr.x;
    outRow[slot] = pr.y;
    if ((slot & 127) == 0) tileMask[tile] = 1ull;
  }
}
// tile -> filter offset table, from the list offsets already on the device (no host round trip)
template <int KMAX>
__global__ void k_deconv_tiles(const int *__restrict__ off, int K, int *__restrict__ tileW, int *__restrict__ tileFirst) {
  __shared__ int first[KMAX + 1];
  if (threadIdx.x == 0) {
    int a = 0;
    for (int k = 0; k < K; k++) { first[k] = a; a += (off[k + 1] - off[k] + 127) / 128; }
    first[K] = a;
  }
  __syncthreads();
  for (int k = 0; k <= K; k++) if (threadIdx.x == 0) tileFirst[k] = first[k];
  for (int k = 0; k < K; k++)
    for (int t = first[k] + threadIdx.x; t < first[k + 1]; t += blockDim.x) tileW[t] = k;
}
// Built on first use by a Deconvolution whose rulebook gives every fine site exactly one parent.
int Metadata::get_deconv_plan(ConvEntry &e) {
  if (!claim(e.deconvRdy)) return 0;
  struct Guard { Metadata &m; Ready &r; ~Guard() { if (!r.ready) m.unclaim(r); } } guard{*this, e.deconvRdy};
  BuildLock bl(*this);
  Grid *gf = find_grid(e.in.data()), *gc = find_grid(e.out.data());
  if (gf) SCN_TRY(need(gf->rdy));
  if (gc) SCN_TRY(need(gc->rdy));
  SCN_TRY(need(e.rdy));
  SCN_CHECK(gf && gc && e.geom.M == 1 && e.rb.total == gf->n, "deconvolution plan needs a single-parent rulebook");
  const int K = e.geom.K, n = gf->n;
  cudaStream_t s = cur().stream;
  // per-offset lists in SPATIAL order of the fine grid (same counts as the reference rulebook)
  int nT = cdiv(std::max(n, 1), kRuleTile);
  int *tileCnt = alloc_n<int>((long)nT * K);
  int2 *dpairs = alloc_n<int2>(std::max(1, n));
  SCN_CHECK(tileCnt && dpairs, "alloc");
  DeconvMask mf{e.geom, gf->p2id, gf->coords};
  DeconvPair pf{e.geom, gf->p2id, gf->coords, view(*gc), gc->p2id};
  if (K > 64) { // one pass per 64 lists (build_rule_lists_wide); the totals are known already (e.rb.off)
    int *totals = alloc_n<int>(K), *tc = alloc_n<int>((long)cdiv(K, 64) * nT * 64);
    SCN_CHECK(totals && tc, "alloc");
    for (int k0 = 0; k0 < K; k0 += 64) {
      const int Lw = std::min(64, K - k0);
      k_rule_count<<<nT, kRuleTile, 0, LS(s)>>>(n, Lw, ChunkMask<DeconvMask>{mf, k0}, tc + (long)(k0 / 64) * nT * 64);
      k_rule_scan<<<Lw, 1024, 0, LS(s)>>>(nT, Lw, tc + (long)(k0 / 64) * nT * 64, totals + k0);
    }
    SCN_TRY(write_rule_lists_wide(*this, n, K, mf, pf, tc, e.rb.d_off, dpairs));
  } else {
    k_rule_count<<<nT, kRuleTile, 0, LS(s)>>>(n, K, mf, tileCnt);
    k_rule_scan<<<K, 1024, 0, LS(s)>>>(nT, K, tileCnt, cur().d_scalars + 128);
    if (n > 0) k_rule_write<<<nT, kRuleTile, 0, LS(s)>>>(n, K, mf, pf, tileCnt, e.rb.d_off, dpairs);
  }
  DeconvPlan &d = e.deconv;
  d.nTiles = 0;
  for (int k = 0; k < K; k++) d.nTiles += cdiv(e.rb.off[k + 1] - e.rb.off[k], 128);
  d.nbr = alloc_n<int>(std::max(1, d.nTiles) * 128l);
  d.outRow = alloc_n<int>(std::max(1, d.nTiles) * 128l);
  d.tileW = alloc_n<int>(std::max(1, d.nTiles));
  d.tileMask = alloc_n<unsigned long long>(std::max(1, d.nTiles) + 8);
  int *dFirst = alloc_n<int>(K + 1);
  SCN_CHECK(d.nbr && d.outRow && d.tileW && d.tileMask && dFirst, "alloc");
  if (d.nTiles) {
    if (K > 64) k_deconv_tiles<kMaxFilterVolume><<<1, 256, 0, LS(s)>>>(e.rb.d_off, K, d.tileW, dFirst);
    else k_deconv_tiles<64><<<1, 256, 0, LS(s)>>>(e.rb.d_off, K, d.tileW, dFirst);
    k_deconv_pad<<<stream_grid(d.nTiles * 128l, 256), 256, 0, LS(s)>>>(dpairs, e.rb.d_off, d.tileW, dFirst, d.nTiles, d.nbr, d.outRow, d.tileMask);
  }
  SCN_CUDA(cudaGetLastError());
  d.built = true;
  SCN_TRY(mark_ready(e.deconvRdy));
  return 0;
}

// ------------------------------------------------------------------ getSpatialLocations
__global__ void k_locations(const int4 *coords, int n, long *out) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int4 c = coords[i];
    out[i * 4 + 0] = c.x; out[i * 4 + 1] = c.y; out[i * 4 + 2] = c.z; out[i * 4 + 3] = c.w;
  }
}
// Metadata::getSpatialLocations (Metadata.cpp:147-168): int64 [nActive][4] in row-id order
int Metadata::spatial_locations(const long *sz, long *out, int outOnDevice) {
  BuildLock bl(*this);
  Grid *g = find_grid(sz);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  if (g->n == 0) return 0;
  SCN_TRY(need(g->rdy));
  long *dst = out;
  if (!outOnDevice) { dst = alloc_n<long>((long)g->n * 4); SCN_CHECK(dst, "alloc"); }
  if (outOnDevice) SCN_TRY(from_compute()); // `out` was allocated by the caller on its cur().stream
  k_locations<<<stream_grid(g->n, 256), 256, 0, LS(cur().stream)>>>(g->coords, g->n, dst);
  SCN_CUDA(cudaGetLastError());
  if (outOnDevice) { Ready r; SCN_TRY(mark_ready(r)); SCN_TRY(wait_ready(r)); }
  if (!outOnDevice) {
    SCN_CUDA(cudaMemcpyAsync(out, dst, (long)g->n * 32, cudaMemcpyDeviceToHost, cur().stream));
    SCN_CUDA(cudaStreamSynchronize(cur().stream));
  }
  return 0;
}

} // namespace scn
