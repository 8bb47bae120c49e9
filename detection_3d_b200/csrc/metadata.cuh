// Device-resident Metadata: per spatial size an active-site grid (block directory + occupancy
// masks for neighbour probes, reference row numbering, reference hash-iteration order) and the
// rulebooks / execution plans derived from it.  Replaces the host-side Metadata<3> of the
// reference (SCN/Metadata/Metadata.h:44-163, Metadata.cpp).
#pragma once
#include "common.cuh"
#include <map>
#include <vector>
#include <array>
#include <mutex>
#include <condition_variable>
#include <chrono>
#include <atomic>
#include <thread>

struct scn_metadata;

namespace scn {

typedef std::array<long, 3> P3;

// `ready` (guarded by Metadata::mapMu) flips once the object is completely described on the host and
// all its kernels are queued on a build stream (`by`); `building` = some thread has claimed the build;
// `ev` marks the end of the build on that stream: other build streams (Metadata::need) and the
// first feature kernel that uses the object (`waited`, Metadata::wait_ready) wait for it.
struct Ready {
  bool ready = false, building = false; cudaEvent_t ev = nullptr; cudaStream_t by = nullptr; bool waited = false;
  bool ahead = false; // rule lists: built by a prefetch worker from a hint (scn_metadata_prefetch kinds 4 / 5), not on demand
};
struct Grid {
  Ready rdy;          // active-site structures (directory, masks, numbering)
  Ready rankRdy;      // rank2id (reference hash-iteration order)
  P3 sz{};            // spatial size
  int n = 0;          // active sites over all batch items (host copy)
  int batch = 1;
  // block directory: 8x8x8 blocks, one directory plane per batch item
  int dd[3] = {0, 0, 0};
  long dirCells = 0;  // per batch item
  int *dir = nullptr;                  // [batch*dirCells] block index or -1
  unsigned long long *bmask = nullptr; // [maxBlocks*8] 512-bit occupancy per block
  int *wbase = nullptr;                // [maxBlocks*8] spatial index of the first bit of each word
  int *d_nblocks = nullptr;            // device scalar
  long maxBlocks = 0;
  int4 *coords = nullptr;              // [n] (x,y,z,batch) by row id  (reference numbering)
  int *p2id = nullptr, *id2p = nullptr; // spatial index <-> row id
  int *rank2id = nullptr;              // reference hash-iteration order (batch items concatenated)
  bool hasRank = false;
  std::vector<int> itemCount;          // sites per batch item (host)
  std::vector<int> itemCtr;            // SparseGrid::ctr per item (id offset); -1 when ids interleave (input grid)
  bool built = false;
};

// One rulebook in the reference's format: nLists lists of (in,out) int32 pairs, concatenated;
// list k occupies pairs [off[k], off[k+1]).
struct RuleBookDev {
  int nLists = 0;
  int2 *pairs = nullptr;      // device
  std::vector<int> off;       // host, nLists+1
  int *d_off = nullptr;       // device copy
  long total = 0;
};

// Output-stationary execution plan: for every output site (in spatial order p) the input row of
// each filter offset, or -1.  Layout: tiles of 128 consecutive sites; inside a tile the 128 ids of
// one filter offset are contiguous (one coalesced 512-byte read per (tile, offset) in the gather
// kernels).  The buffer is padded with -1 to whole work items of kPlanPad sites.
struct NbrPlan {
  int K = 0;
  int nOut = 0;
  int *nbr = nullptr;         // [plan_padded(nOut)*K] input row ids at nbr_index(p, k, K), p = OUTPUT spatial index
  const int *outRow = nullptr; // p -> output row id (p2id of the output grid)
  const int *slot = nullptr;  // optional: plan slot of spatial index p (sorted plans, get_submanifold); null = slot p
  long nValid = 0;            // number of non-negative entries (= rules)
  unsigned long long *tileMask = nullptr; // per 128-site tile: bit k set when some site of the tile has a neighbour at offset k
};

struct SubmKey { P3 sz, f; bool operator<(const SubmKey &o) const { return sz != o.sz ? sz < o.sz : f < o.f; } };
struct ConvKey { P3 in, f, s; bool operator<(const ConvKey &o) const { return in != o.in ? in < o.in : (f != o.f ? f < o.f : s < o.s); } };

// Deconvolution plan (single-parent strided rulebooks): fine sites grouped by filter offset, each group
// padded to whole 128-row tiles, so that one tile needs exactly one weight slice.
struct DeconvPlan {
  bool built = false;
  int nTiles = 0;
  int *nbr = nullptr;      // [nTiles*128] coarse (source) row or -1 (padding)
  int *outRow = nullptr;   // [nTiles*128] fine (destination) row or -1
  int *tileW = nullptr;    // [nTiles] weight slice (filter offset) of the tile
  unsigned long long *tileMask = nullptr; // [nTiles] all ones (kept for the kernel's interface)
};
struct ConvGeomHost { int f[3], s[3], outS[3], cnt[3], M, K; };
struct SubmEntry { RuleBookDev rb; NbrPlan plan; Ready rdy, rulesRdy; P3 sz; bool assigned = false; /* the second prefetch worker will build it */ }; // rb.pairs / offsets only after ensure_subm_rules
// rb.pairs (the (in,out) lists in the reference's order) are written on demand (ensure_conv_rules: backward pass, rulebook
// inspection, CUDA-core deconvolution); the forward needs only the plan, the list offsets and the rule count.
struct ConvEntry {
  RuleBookDev rb; NbrPlan plan; P3 out; P3 in; ConvGeomHost geom; DeconvPlan deconv; Ready rdy, deconvRdy, rulesRdy;
  const int *evQ = nullptr; int *tileCnt = nullptr; // kept for the deferred list write
  bool gridGiven = false; // the output grid and evQ came from overlay_conv: get_conv builds the lists and the plan over that grid
};

struct InputRules {
  int mode = 0, maxActive = 0, nIn = 0, nOut = 0;
  int *tab = nullptr;  // [nOut*(1+maxActive)] device
  // per input row: spatial index and coordinates; per site (spatial index): first / last input row (lastRow: mode 2 only).
  // Numbering-independent: overlay_input numbers a twin's input level from them.
  const int *rowP = nullptr, *firstRow = nullptr, *lastRow = nullptr;
  const int4 *pts = nullptr;
  bool valid = false;
  Ready rdy;
};

struct Chunk { void *p; size_t cap; cudaEvent_t freed; };
// Everything a thread needs to BUILD (grids, hash order, rulebooks, plans): a private high-priority
// stream, scalar scratch with its pinned host mirror, zeroed scan state and a bump allocator.  The
// caller's thread and the chain worker share context 0, the second prefetch worker owns context 1.
struct BuildCtx {
  cudaStream_t stream = 0;
  bool ownStream = false;
  bool lowPrio = false;     // stream taken from the normal-priority list (use_low_priority_streams)
  int *d_scalars = nullptr; // small device scratch (256 ints)
  int *h_scalars = nullptr; // pinned host mirror
  int *d_err = nullptr;
  unsigned long long *zpool = nullptr; // zero-initialised pool for scan states
  size_t zpoolWords = 0, zpoolUsed = 0;
  // bump allocator over a few chunks: a Metadata makes ~350 small allocations per forward and frees them all together
  char *arena = nullptr;
  size_t arenaCap = 0, arenaUsed = 0, arenaNext = 16u << 20;
  std::vector<Chunk> chunks; // device memory taken from the process-wide list, returned on destruction
  std::recursive_mutex mu;   // serialises the builds that use this context
  // glibc mutexes are not fair: a worker that re-locks `mu` for its next entry right after unlocking
  // starves the caller (measured: the caller's first convolution waited 5.8 ms, until the worker had
  // built the whole pyramid).  The caller announces itself here and the worker yields.
  std::atomic<int> callerWaiting{0};
};
struct Metadata {
  // Feature kernels run on the caller's `cstream`; builds (many short kernels and a few host
  // readbacks of counts) run on the private streams of the build contexts, so a host wait for a count
  // only drains a short build queue while the convolutions already submitted keep the GPU busy (the
  // reference is synchronous throughout, SURVEY.md section 8b "Threading / streams").
  cudaStream_t cstream = 0;  // caller's compute stream
  // Internal numbering (program replay only, never exposed): row id = spatial index.  Skips the emulation of the reference's
  // hash-iteration order and the first-touch numbering -- the two steps that serialise the grid pyramid; the reference
  // numbering of the few OUTPUT levels comes from a second, ordinary Metadata built beside it (program.cu).
  bool spatialIds = false;
  bool poolGrowth = false;   // may take fresh memory instead of waiting for chunks a running forward still owns
  BuildCtx cx[2];
  int nCtx = 1;
  BuildCtx &cur();           // build context of the calling thread
  cudaEvent_t evCompute = nullptr;
  int use_low_priority_streams(); // builds of this Metadata are not urgent: move its build contexts to normal-priority streams
  int from_compute();        // the current build stream waits for everything the caller has queued so far
  void to_compute();         // the caller's stream waits for everything the build streams have queued so far
  // `mapMu` guards the structure of the caches and the ready / building flags; `cv` wakes threads
  // that wait for an entry another thread is building.
  std::mutex mapMu;
  std::condition_variable cv;
  std::atomic<bool> chainDone{true}; // no chain worker is producing grids (set_chain_done)
  std::atomic<bool> worker2Done{true}; // the second prefetch worker is not running (entries marked `assigned` will not be built by it)
  std::vector<cudaEvent_t> events;
  struct BuildLock {
    BuildCtx &c;
    explicit BuildLock(Metadata &md);
    ~BuildLock() { c.mu.unlock(); }
  };
  bool claim(Ready &r);       // false: already built; true: the caller builds it (others wait in claim)
  void unclaim(Ready &r);     // a build failed: let a waiter retry
  int mark_ready(Ready &r);   // record r.ev on the current build stream, publish r.ready
  int need(Ready &r);         // the current build stream waits for something built on another build stream
  int wait_ready(Ready &r);   // first use on the compute stream: wait for r.ev
  bool is_ready(const Ready &r) { std::lock_guard<std::mutex> lk(mapMu); return r.ready; }
  Grid *find_grid_wait(const long *sz);
  ConvEntry *wait_conv(const long *inS, const long *f, const long *st);
  void set_chain_done(bool v);
  std::map<P3, Grid> grids;
  std::map<SubmKey, SubmEntry> subm;   // submanifoldRuleBooks, Metadata.h:58-60
  std::map<ConvKey, ConvEntry> conv;   // ruleBooks, Metadata.h:65-67
  InputRules input;

  ~Metadata();
  int init();
  void *alloc(size_t bytes);
  void *alloc_in(BuildCtx &c, size_t bytes);
  template <class T> T *alloc_n(size_t n) { return static_cast<T *>(alloc(n * sizeof(T) + 16)); }
  unsigned long long *scan_state(long n);
  int sync_scalars(int count);

  int input_layer(const long *sz, const long *coords, int coordsOnDevice, long nrows, int ncols,
                  int batchHint, int mode);
  int input_rules(const Grid &g);
  // Reference numbering over the grids of an internally numbered Metadata `in` built from the same input (one batch item):
  // the input level, and the output grid of one strided convolution, take the block structure of `in`'s grid of the same
  // size and compute only the reference row ids (and the hash-iteration order that induces them).
  int overlay_input(Metadata &in, const long *sz);
  int overlay_conv(Metadata &in, const long *inS, const long *outS, const long *f, const long *st);
  Grid *find_grid(const long *sz);
  int ensure_rank(Grid &g);
  int get_submanifold(const long *sz, const long *f, SubmEntry **out);
  int ensure_subm_rules(SubmEntry &e, bool ahead = false); // ahead: called by a prefetch worker (Ready::ahead)
  int get_conv(const long *inS, const long *outS, const long *f, const long *s, ConvEntry **out);
  int get_conv_small(Grid &gi, Grid &go, ConvEntry &e, const ConvGeomHost &G); // one-launch build for small input grids
  int ensure_conv_rules(ConvEntry &e, bool ahead = false);
  int spatial_locations(const long *sz, long *out, int outOnDevice);
  int build_tile_masks(NbrPlan &plan);
  int get_deconv_plan(ConvEntry &e);
};
int build_subm_on_caller(Metadata &md, const long *sz, const long *f);
void set_prefetch_worker_thread(bool on, int ctx);
// the process-wide chunk pool (scn_set_pool_growth, scn_debug_counter(0..2), scn_release_cached_memory)
void set_pool_growth(int on);
long debug_chunk_mallocs();
long debug_chunk_waits();
long debug_chunk_total_mb();
long release_idle_chunks();
Metadata *metadata_of(scn_metadata *m); // (capi.cu)

// ------------------------------------------------------------------ device helpers
__host__ __device__ __forceinline__ uint32_t point_hash(int x, int y, int z) {
  // IntArrayHash<3>, SCN/Metadata/32bits.h:57-66
  uint32_t h = 16777619u;
  h *= 2166136261u; h ^= (uint32_t)x;
  h *= 2166136261u; h ^= (uint32_t)y;
  h *= 2166136261u; h ^= (uint32_t)z;
  return h;
}

struct GridView {
  const int *dir;
  const unsigned long long *bmask;
  const int *wbase;
  int dd0, dd1, dd2;
  long dirCells;
  int sz0, sz1, sz2;
};
// occupancy test only (no rank): is (x, y, z, b) an active site?
__device__ __forceinline__ bool grid_has(const GridView &g, int x, int y, int z, int b) {
  if ((unsigned)x >= (unsigned)g.sz0 || (unsigned)y >= (unsigned)g.sz1 || (unsigned)z >= (unsigned)g.sz2) return false;
  long cell = (long)b * g.dirCells + ((long)(x >> 3) * g.dd1 + (y >> 3)) * g.dd2 + (z >> 3);
  int blk = __ldg(g.dir + cell);
  if (blk < 0) return false;
  int bit = ((x & 7) << 6) | ((y & 7) << 3) | (z & 7);
  return (__ldg(g.bmask + blk * 8 + (bit >> 6)) >> (bit & 63)) & 1ull;
}
// spatial index of an active site, or -1
__device__ __forceinline__ int grid_lookup(const GridView &g, int x, int y, int z, int b) {
  if ((unsigned)x >= (unsigned)g.sz0 || (unsigned)y >= (unsigned)g.sz1 || (unsigned)z >= (unsigned)g.sz2) return -1;
  long cell = (long)b * g.dirCells + ((long)(x >> 3) * g.dd1 + (y >> 3)) * g.dd2 + (z >> 3);
  int blk = __ldg(g.dir + cell);
  if (blk < 0) return -1;
  int bit = ((x & 7) << 6) | ((y & 7) << 3) | (z & 7);
  int w = blk * 8 + (bit >> 6);
  unsigned long long m = __ldg(g.bmask + w);
  unsigned long long one = 1ull << (bit & 63);
  if (!(m & one)) return -1;
  return __ldg(g.wbase + w) + __popcll(m & (one - 1));
}

} // namespace scn
