// Shared device/host utilities for the B200 sparse-convolution library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <atomic>

namespace scn {

// ---------------------------------------------------------------- errors
void set_error(const std::string &msg);
const char *last_error(); // this thread's last message
#define SCN_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      char b__[512];                                                                     \
      snprintf(b__, sizeof b__, "%s:%d %s -> %s", __FILE__, __LINE__, #call,             \
               cudaGetErrorString(e__));                                                 \
      scn::set_error(b__);                                                               \
      return -1;                                                                         \
    }                                                                                    \
  } while (0)
#define SCN_CHECK(cond, msg)                                                             \
  do {                                                                                   \
    if (!(cond)) {                                                                       \
      char b__[512];                                                                     \
      snprintf(b__, sizeof b__, "%s:%d check failed: %s (%s)", __FILE__, __LINE__, #cond, msg); \
      scn::set_error(b__);                                                               \
      return -2;                                                                         \
    }                                                                                    \
  } while (0)
#define SCN_TRY(expr)                                                                    \
  do {                                                                                   \
    int r__ = (expr);                                                                    \
    if (r__ != 0) return r__;                                                            \
  } while (0)

// developer timeline (SCN_TIMELINE=1): host timestamps of build / submit milestones, printed to stderr
void timeline_mark(const char *who, int kind, long a, long b);
void timeline_dump();
// every kernel launch of this library passes its stream through LS(): launch accounting
extern std::atomic<long> g_launches;
static inline cudaStream_t LS(cudaStream_t s) { ++g_launches; return s; }
// which-fusion-was-taken counters (scn_debug_counter(3..)): the parity tests assert on them that the benchmarked code path
// -- lateral stage, epilogue statistics, bf16-only outputs -- really ran, instead of a silent fallback
enum DebugCounter {
  kCntLateralFolded = 3,   // tensor-core launches that carried a lateral 1x1x1 stage (in2 / wimg2)
  kCntEpilogueStats = 4,   // tensor-core launches whose epilogue accumulated BatchNorm statistics
  kCntHalfOnlyOut = 5,     // program registers that were written as bf16 only (no fp32 rows)
  kCntLateralFallback = 6, // laterals the program executor had to run as a separate 1x1x1 convolution + add
  kCntTcLaunch = 7,        // conv_plan_tc launches
  kCntBnFromSums = 8,      // BatchNorm ops that ran their apply pass from epilogue statistics
  kCntSplitLaunch = 9,     // conv_plan_tc launches that split the filter offsets over CTAs (atomic epilogue)
  kCntSimtLaunch = 10,     // CUDA-core convolution launches (plan or list)
  kCntTrainReplay = 11,    // backward passes run by the program executor (scn_program_backward)
  kCntDwPlanLaunch = 13,   // weight-gradient launches driven by the output-stationary plan (conv_dw_plan_tc)
  kCntBwdOperandReused = 12, // bf16 operand copies the weight-gradient kernel took from its caller instead of converting again
  kCntFloatAtomic = 14,    // launches that accumulated floats with atomics, i.e. whose result depends on the order the atomics land in
  kCntTf32x3Launch = 15,   // conv_plan_tc launches with TF32X3 operands (math mode 3)
  kCntChunkedLaunch = 16,  // conv_plan_tc launches over one offset chunk of a plan with more than 64 filter offsets
  kCntCoordUpload = 17,    // host -> device copies of input-layer coordinates
  kCntF16Launch = 18,      // tensor-core launches with fp16 operands (math mode 5): conv_plan_tc and the weight-gradient kernels
  kCntRulesAhead = 19,     // rule lists a backward entry found already built (hinted ahead by a training run, program.cu)
  kCntTrainPrepared = 20,  // training runs that took a Metadata prepared by scn_program_prepare_training
  kCntSimtDwLaunch = 21,   // CUDA-core weight-gradient launches of the sparse convolutions (k_dw, one per rule list)
  kCntDwX3Launch = 22,     // weight-gradient launches with three-way bf16 operand splits (conv_dw_tc, math mode 3)
  kCntCounters = 23
};
extern std::atomic<long> g_counters[kCntCounters];

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------- deterministic mode (scn_set_deterministic)
// On: every launcher that would accumulate floats with atomics writes per-work-item partials to fixed slots instead and sums them
// in index order, so that results do not depend on which CTA ran first.  Read at launch time.
bool deterministic();
// grow-only scratch of the deterministic mode's partial sums, one per (device, stream); uses on one stream are ordered
int det_scratch(cudaStream_t s, size_t bytes, void **out);
// out[map(j)] = sum over p = 0 .. nPart-1 of part[p * width + j] for j < width, in an order fixed by (nPart, width) alone;
// map(j) = j, or (j / seg) * segStride + j % seg when seg > 0.  T = float or double (accumulated in double).
template <class T>
int ordered_sum(const T *part, int nPart, long width, T *out, cudaStream_t s, long seg = 0, long segStride = 0);

// ---------------------------------------------------------------- 16-bit operand modes (scn_set_math_mode)
// Math modes 2 (bf16) and 5 (fp16) give the tensor cores 16-bit operands on the same layers: rows of a multiple of 64 channels
// and the packed 16- / 32-channel rows; the other layers keep TF32 operands.  Every 16-bit copy of a feature matrix -- the
// "bf16" arguments of the C ABI, the shadows of a recorded program, the operand copies the launchers make -- is written and read
// in the format of the current mode: fp16 in mode 5, bf16 in every other mode (as before mode 5 existed).
constexpr int kModeBF16 = 2, kModeTF32X3 = 3, kModeF16 = 5;
static inline bool half_mode(int mathMode) { return mathMode == kModeBF16 || mathMode == kModeF16; }
int math_mode(); // the current mode (capi.cu)
static inline bool f16_copies() { return math_mode() == kModeF16; }
#if defined(__CUDACC__)
} // namespace scn
#include <cuda_bf16.h>
#include <cuda_fp16.h>
namespace scn {
// fp32 -> 16 bits, round to nearest even; fp16 overflows to +-inf (no saturation) and keeps subnormals, as torch's .half() does
template <bool F16>
__device__ __forceinline__ unsigned short to16(float x) {
  if (F16) return __half_as_ushort(__float2half_rn(x));
  return __bfloat16_as_ushort(__float2bfloat16_rn(x));
}
template <bool F16>
__device__ __forceinline__ unsigned int pack16x2(float a, float b) {
  if (F16) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<unsigned int *>(&h); }
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<unsigned int *>(&h);
}
template <bool F16>
__device__ __forceinline__ uint2 pack16x4(float4 v) {
  uint2 pk;
  pk.x = pack16x2<F16>(v.x, v.y);
  pk.y = pack16x2<F16>(v.z, v.w);
  return pk;
}
#endif

// ---------------------------------------------------------------- programmatic dependent launch (sm_90+)
// The layer kernels of a forward sit back to back on one stream, ~100 of them, half of them a few microseconds long.  Launched with
// the programmatic-stream-serialization attribute a kernel's CTAs become resident while the previous kernel is still draining
// and run their prologue (barrier initialisation, TMEM allocation, scale / shift tables); `pdl_wait()` then blocks until the
// previous kernel has completed and its writes are visible.  Rules: (1) a kernel launched through launch_pdl() executes
// pdl_wait() in every thread before its first global-memory access; (2) it calls pdl_launch_dependents() on entry, so that the
// NEXT kernel may do the same (all grids here fit in one wave, so early residents never starve their predecessor's CTAs).
// Any other operation between two kernels (event wait, memset, a kernel launched the ordinary way) keeps full serialisation.
#if defined(__CUDACC__)
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// (the fence makes ptxas emit CCTL.IVALL: an early-resident CTA shares its SM's L1 with CTAs of older kernels that may have cached
//  lines of a buffer the previous kernel has since rewritten -- register buffers are recycled -- and this kernel reads with ld.global.nc)
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n\tfence.acq_rel.gpu;" ::: "memory"); }
#endif
int pdl_mode(); // SCN_PDL: 0 = attribute off (the two instructions are then no-ops), 1 = every launch_pdl() launch, 2 = only grids of at most 64 CTAs
template <class... KArgs, class... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  const int mode = pdl_mode();
  cfg.numAttrs = (mode == 1 || (mode == 2 && (long)grid.x * grid.y * grid.z <= 64)) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// B200: 148 SMs.  Element-wise / streaming kernels use grid-stride loops over a grid that is
// a multiple of the SM count.
constexpr int kSMs = 148;
constexpr int kBnMaxC = 4096; // BatchNorm forward workspace: kBnReplicas x 2*kBnMaxC doubles (statistics) + 2*kBnMaxC floats (scale, shift)
constexpr int kBnReplicas = 8;
constexpr int kFusedStatsC = 128; // channel stride of the statistics a convolution epilogue accumulates: [kBnReplicas][2][kFusedStatsC] doubles
constexpr size_t kBnWorkspaceBytes = (size_t)kBnReplicas * 2 * kBnMaxC * 8 + 2 * kBnMaxC * 4 + 64;
static inline int stream_grid(long n, int threads, int per_sm = 8) {
  long want = (n + threads - 1) / threads;
  long cap = (long)kSMs * per_sm;
  if (want < 1) want = 1;
  return (int)(want < cap ? want : cap);
}

// ---------------------------------------------------------------- execution-plan layout
// (see NbrPlan in metadata.cuh) tiles of 128 output sites, ids of one filter offset contiguous
constexpr int kPlanPad = 512;
__host__ __device__ __forceinline__ long nbr_index(long p, int k, int K) { return ((p >> 7) * K + k) * 128 + (p & 127); }
__host__ __device__ __forceinline__ long plan_padded(long n) { return (n + kPlanPad - 1) / kPlanPad * kPlanPad; }
// Wide plans (K > 64 filter offsets, up to kMaxFilterVolume) are stored CHUNK-MAJOR: chunk c holds offsets [63 c, 63 c + Kc),
// Kc = min(63, K - 63 c), as an ordinary plan of Kc offsets over the same nPad = plan_padded(nOut) sites, at nbr + 63 c nPad; its
// per-tile offset masks (bit j = offset 63 c + j) are at tileMask + c nPad / 128.  A chunk is then exactly what the tensor-core
// kernel takes, with bit 63 of its masks left free for the lateral stage.  Plans of K <= 64 keep the single-chunk layout above.
constexpr int kMaxFilterVolume = 512;
constexpr int kChunkOffsets = 63;
__host__ __device__ __forceinline__ int plan_chunks(int K) { return K <= 64 ? 1 : (K + kChunkOffsets - 1) / kChunkOffsets; }
__host__ __device__ __forceinline__ long nbr_index_wide(long p, int k, int K, long nPad) {
  const int c = k / kChunkOffsets, k0 = c * kChunkOffsets, Kc = K - k0 < kChunkOffsets ? K - k0 : kChunkOffsets;
  return (long)k0 * nPad + nbr_index(p, k - k0, Kc);
}

// ---------------------------------------------------------------- single-pass scan
// Decoupled look-back exclusive scan (int32) with a fused consumer.  One launch:
//   value_i  = in(i)
//   out(i, exclusive_prefix_i, value_i)
//   *total   = sum (optional)
// `state` must point at zero-initialised memory: [0] tile ticket, then one uint64 status word
// per tile ((flag << 32) | value, flag 1 = aggregate, 2 = inclusive prefix).
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

static inline size_t scan_state_words(long n) { return 2 + (size_t)((n + kScanTile - 1) / kScanTile); }

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += t;
  }
  return v;
}

template <class InF, class OutF>
__global__ void __launch_bounds__(kScanThreads) scan_kernel(long n, InF in, OutF out,
                                                            unsigned long long *state, int *total) {
  __shared__ int s_warp[kScanThreads / 32];
  __shared__ int s_tile, s_prefix;
  unsigned int *ticket = reinterpret_cast<unsigned int *>(state);
  volatile unsigned long long *status = state + 1;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_tile = (int)atomicAdd(ticket, 1u);
  __syncthreads();
  const int tile = s_tile;
  const long base = (long)tile * kScanTile + (long)tid * kScanItems;
  int v[kScanItems];
  int sum = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; j++) {
    long i = base + j;
    v[j] = i < n ? in(i) : 0;
    sum += v[j];
  }
  int incl = warp_incl_scan(sum, lane);
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int w = lane < kScanThreads / 32 ? s_warp[lane] : 0;
    int wi = warp_incl_scan(w, lane);
    if (lane < kScanThreads / 32) s_warp[lane] = wi - w; // exclusive prefix of each warp
    const int tile_sum = __shfl_sync(0xffffffffu, wi, kScanThreads / 32 - 1);
    // publish aggregate, then look back
    int prefix = 0;
    if (tile == 0) {
      if (lane == 0) status[0] = (2ull << 32) | (unsigned int)tile_sum;
    } else {
      if (lane == 0) status[tile] = (1ull << 32) | (unsigned int)tile_sum;
      int look = tile - 1;
      while (true) {
        int idx = look - lane;
        unsigned long long s = 0;
        if (idx >= 0) {
          do { s = status[idx]; } while ((s >> 32) == 0);
        } else {
          s = (2ull << 32); // virtual tile before 0: inclusive prefix 0
        }
        const unsigned flag = (unsigned)(s >> 32);
        const int val = (int)(unsigned)s;
        const unsigned incl_mask = __ballot_sync(0xffffffffu, flag == 2);
        // lanes closer than the first inclusive-prefix lane contribute aggregates
        const int first = incl_mask ? __ffs(incl_mask) - 1 : 32;
        int contrib = (lane <= first) ? val : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
        prefix += contrib;
        if (incl_mask) break;
        look -= 32;
      }
      if (lane == 0) status[tile] = (2ull << 32) | (unsigned int)(prefix + tile_sum);
    }
    if (lane == 0) {
      s_prefix = prefix;
      if (total && (long)(tile + 1) * kScanTile >= n) *total = prefix + tile_sum;
    }
  }
  __syncthreads();
  int run = s_prefix + s_warp[wid] + (incl - sum);
#pragma unroll
  for (int j = 0; j < kScanItems; j++) {
    long i = base + j;
    if (i < n) out(i, run, v[j]);
    run += v[j];
  }
}

} // namespace scn
