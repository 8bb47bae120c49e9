// tcgen05 tensor-core gather-GEMM for sm_100a: the output-stationary sparse convolution
//   out[row(p)] = sum_k  in[nbr[p][k]] @ W[k]
// with fp32 accumulators in TMEM across ALL filter offsets (one store per output element, no
// read-modify-write, no atomics).
//
// Persistent kernel, one CTA per SM, warp-specialised (14 warps):
//   warps 0-3   epilogue   (tcgen05.ld -> registers -> shared-memory transpose -> 128-byte row stores)
//   warps 4-11  A producers (16-byte cp.async row gathers into 128B-swizzled K-major atoms)
//   warp  12    MMA issuer (one thread: tcgen05.mma M=128, N=Cout, 32 bytes of K per instruction)
//   warp  13    B loader   (one thread: cp.async.bulk of a pre-swizzled weight atom)
//
// Work item  = T <= 4 tiles of 128 output sites (x a range of filter offsets on small levels).
// Stage      = one 128-byte K atom (32 tf32 / 64 bf16 channels) of ONE filter offset for ALL T tiles
//              (T x 16 KB of gathered rows) + the matching weight atom (Cout x 128 B).
// What was measured on B200 and shaped this (profiles/r1_conv_tc_design_notes.md):
//   * the issuing thread pays ~400 cycles per barrier round trip (try_wait + fence + commit), so a
//     stage must carry >= ~1000 cycles of MMA: 4 tiles x 4 MMAs x 64 cycles; one full and one
//     empty barrier per stage shared by the A and B halves;
//   * the weight atom is read once per stage and feeds T tiles: L2->SM traffic of W is 1/T of a
//     per-tile scheme (with T = 2 it equalled the gather traffic);
//   * TMA tile::gather4 delivers correct swizzled rows but only ~7.5 B/clk/SM at 128-byte rows,
//     against ~32 B/clk/SM for 16-byte cp.async, hence cp.async gathers.
//
// Replaces dConvolution_KMxKN_forwardA/B (SCN/CUDA/Convolution.cu:57-203: SIMT tiles, fp64
// accumulators, one launch + one blocking H2D rule copy per filter offset).
#include "conv.cuh"
#include <cuda_bf16.h>
#include <stdlib.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

namespace scn {

constexpr int kTileM = 128;
constexpr int kAtomBytes = kTileM * 128; // 128 rows x 128 B
constexpr int kMaxT = 4;
constexpr int kLateralBit = 63; // mask bit of the lateral stage (launches with a lateral stage have K <= 63; a K = 64 plan uses bit 63 for offset 63)
#ifndef SCN_EPI_COLS
#define SCN_EPI_COLS 32
#endif
constexpr int kEpiCols = SCN_EPI_COLS;           // output columns per epilogue round: 32 (16 KB of staging per CTA) or 16 (8 KB)
constexpr int kEpiBytes = 4 * 32 * kEpiCols * 4; // 4 epilogue warps x (32 rows x kEpiCols floats), XOR-swizzled
constexpr int kBuildRoom = SCN_EPI_COLS == 16 ? 12 * 1024 : 0; // shared memory per SM left to the build kernels that run beside this one
// Operand type of conv_plan_tc (template parameter OP).  TF32X3 ("3xTF32", math mode 3): every fp32 operand x = hi + lo with
// both parts exact TF32 values, and out += A_hi W_lo + A_lo W_hi + A_hi W_hi in the same fp32 accumulator (the dropped
// A_lo W_lo and the rounding of lo leave ~2^-21 relative error per product).  F16 (math mode 5): fp16 operands wherever bf16 mode
// has bf16 ones -- the same kind::f16 instruction and the same 2-byte rows, only the A / B format field of the instruction
// descriptor differs (F16 = 0, BF16 = 1).
enum TcOperand { kOpTF32 = 0, kOpBF16 = 1, kOpTF32X3 = 2, kOpF16 = 3 };
constexpr int kSplitWarps = 4; // TF32X3: warps that split the gathered A atoms of a stage into hi / lo parts

struct TcParams {
  const unsigned char *in; // activations, row-major, rowBytes per row (fp32 or bf16 elements)
  float *out;
  const unsigned char *wimg;
  const float *bias;
  const float *addend; // optional [output rows][Cout]: out = conv + addend (the residual / lateral add fused into the epilogue)
  void *out16;         // optional 16-bit copy of the result (gather operand of the next convolution in bf16 / fp16 mode): bf16, fp16 with OP F16
  const int *nbr;
  const int *outRow;
  const unsigned long long *tileMask;
  const int *tileW; // optional: weight slice per tile (deconvolution plans; then K == 1 and T == 1)
  // optional second source ("lateral"): out += in2[outRow] @ W2, one more accumulation stage per tile, carried as pseudo filter offset kLateralBit
  const unsigned char *in2, *wimg2;
  int rowBytes2, nAtoms2;
  double *stats;    // optional [kBnReplicas][2][kFusedStatsC]: per-channel sum / sum of squares of `out` (statistics of a following BatchNorm)
  long long *prof;  // developer: per-CTA stall counters (SCN_TC_PROF)
  int nOut, K, Cout, ldo, nTiles, // ldo: row stride (elements) of out, addend and out16 -- Cout, or the full width of a column slab's rows
      T, nSuper, S, nAcc, lag;
  int rowBytes, nAtoms, bf16, tmemCols;
  int KG;     // packed layers (template G > 1): number of offset groups = ceil(K / G)
  int dbg;    // developer switches (SCN_TC_DBG): 1 = skip A gathers, 2 = skip B copies, 4 = skip MMAs
  int kSplit; // > 1: the filter offsets of a work item are split over kSplit CTAs, epilogue accumulates atomically
  unsigned *sched; // dynamic work distribution: [0] next work item, [1] CTAs that have drawn their last item (self-resetting); null = static stride
  double *statsPart; // deterministic mode, with stats: [work item][epilogue warp][2][Cout] per-item sums instead of atomics into `stats`
  float *part;       // deterministic mode, kSplit > 1: [kSplit][nOut][Cout] per-split partial outputs instead of atomics into `out`
  int f16;           // OP TF32 only: out16 is fp16 (a narrow layer that keeps TF32 operands in fp16 mode), else bf16
};

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, long long &acc, bool on) {
  if (!on) { mbar_wait(bar, parity); return; }
  long long t0 = clock64();
  mbar_wait(bar, parity);
  acc += clock64() - t0;
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t srcBytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(srcBytes) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ bool elect_one() { // one lane of the (converged) warp
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
template <bool BF16>
__device__ __forceinline__ void tc_mma(uint32_t dTmem, uint64_t aDesc, uint64_t bDesc, uint32_t idesc, uint32_t accumulate) {
  if (BF16)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(dTmem),
        "l"(aDesc), "l"(bDesc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(dTmem),
        "l"(aDesc), "l"(bDesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// fp32 -> the nearest TF32 value (ties away from zero), as an fp32 number whose low 13 mantissa bits are zero
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r & 0xffffe000u);
}
// x = hi + lo, hi = tf32(x), lo = tf32(x - hi) (x - hi is exact in fp32)
__device__ __forceinline__ void tf32_split(float x, float &hi, float &lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);
}
// K-major, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (SBO), version 1 (sm_100)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
      "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
        "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned long long range_mask(int lo, int hi) { // bits [lo, hi)
  unsigned long long a = hi >= 64 ? ~0ull : ((1ull << hi) - 1ull);
  return a & ~((1ull << lo) - 1ull);
}

// the part of a work item every role needs: tiles, offset range, per-tile masks
struct Item {
  int st, part;
  unsigned long long m[kMaxT], uni;
};
// G > 1 (packed layers, rows of 128 / G bytes): G consecutive filter offsets share one 128-byte K atom.  The
// masks then carry one bit per GROUP, kept at bit position G * group (so that `k` in the role loops is the first
// offset of the group); a group is live when any of its offsets is.
template <int G>
__device__ __forceinline__ unsigned long long group_mask(unsigned long long m) {
  if (G == 2) return (m | (m >> 1)) & 0x5555555555555555ull;
  if (G == 4) return (m | (m >> 1) | (m >> 2) | (m >> 3)) & 0x1111111111111111ull;
  return m;
}
template <int G>
__device__ __forceinline__ Item load_item(const TcParams &P, int wi) {
  Item I;
  I.st = wi / P.kSplit;
  I.part = wi - I.st * P.kSplit;
  const int nG = G > 1 ? P.KG : P.K; // split whole groups over the CTAs of an item
  const unsigned long long kmask = range_mask(G * (nG * I.part / P.kSplit), G * (nG * (I.part + 1) / P.kSplit));
  I.uni = 0;
#pragma unroll
  for (int t = 0; t < kMaxT; t++) {
    const int tile = I.st * P.T + t;
    // (no plan = dense rows, NetworkInNetwork: the one "filter offset" is live everywhere)
    I.m[t] = (t < P.T && tile < P.nTiles) ? (group_mask<G>(P.tileMask ? __ldg(P.tileMask + tile) : 1ull) & kmask) : 0ull;
    if (G == 1 && P.in2 && I.part == 0 && t < P.T && tile < P.nTiles) I.m[t] |= 1ull << kLateralBit;
    I.uni |= I.m[t];
  }
  return I;
}

// whether mask bit k of a work item is the lateral stage: only in a launch that carries one (a plan with K = 64 uses bit 63 for its
// last filter offset; the launcher folds a lateral stage into plans with K < 64 only)
__device__ __forceinline__ bool is_lateral(const TcParams &P, int k) { return k == kLateralBit && P.in2 != nullptr; }

// ------------------------------------------------------------------ dynamic work distribution
// Work items are handed out by a global counter instead of a static stride: a CTA that starts late (its SM was still running a
// kernel of another stream -- the rulebook builds run beside the layers) or draws long items simply takes fewer of them, so the
// launch ends when the work ends instead of when the unluckiest CTA ends.  One thread per CTA (the weight loader) draws the
// items, one ahead of its own use, and publishes them to the other roles through a 4-slot ring in shared memory
// (full / empty mbarriers): every role sees the same item sequence.
constexpr int kSchedSlots = 4;
struct Sched {
  uint64_t *full, *empty; // [kSchedSlots]
  volatile int *item;     // [kSchedSlots]
};
// consumer side: item number n of this CTA (or -1: no more work).  Called by whole warps or by a single thread.
__device__ __forceinline__ int sched_take(const Sched &S, int n, bool arrive) {
  const int slot = n & (kSchedSlots - 1);
  mbar_wait(smem_u32(S.full + slot), (uint32_t)(n / kSchedSlots) & 1u);
  const int wi = S.item[slot];
  __syncwarp(__activemask());
  if (arrive) mbar_arrive(smem_u32(S.empty + slot));
  return wi;
}
// producer side (one thread)
__device__ __forceinline__ int sched_draw(const TcParams &P, int nWork) {
  const unsigned v = atomicAdd(P.sched, 1u);
  if (v < (unsigned)nWork) return (int)v;
  if (atomicAdd(P.sched + 1, 1u) == gridDim.x - 1) { P.sched[0] = 0u; P.sched[1] = 0u; } // every CTA draws exactly one item beyond the end: the last one resets the counters
  return -1;
}
__device__ __forceinline__ void sched_publish(const Sched &S, int n, int wi) {
  const int slot = n & (kSchedSlots - 1);
  if (n >= kSchedSlots) mbar_wait(smem_u32(S.empty + slot), (uint32_t)(n / kSchedSlots - 1) & 1u);
  S.item[slot] = wi;
  mbar_arrive(smem_u32(S.full + slot)); // (mbarrier arrive has release semantics at CTA scope: the store above is visible to the waiters)
}

// ------------------------------------------------------------------ kernel
// Launch bound 576 (> the 448 threads used) caps the kernel at 112 registers per thread: a resident
// CTA then leaves ~15K registers and ~17 KB of shared memory per SM, enough for the short
// rulebook-build kernels of the other stream to run beside it instead of queueing behind it.
// PW = producer warps: 8 with one CTA per SM (all 512 TMEM columns), 4 with two CTAs per SM (256
// columns and half the shared memory each): two independent pipelines per SM hide each other's
// barrier hand-offs.
// CTAS = CTAs per SM the variant is built for (register cap: 65536 / (CTAS x threads)): <PW 8, CTAS 2> caps the kernel at 72
// registers (a few spilled words in the epilogue) and doubles the gather issue rate of the two-CTA configuration.
// DET = deterministic mode (P.part / P.statsPart may be set): a separate instantiation, so that the default kernels stay as they are.
// OP = operand type (TcOperand).  TF32X3 is built for the one-CTA configuration only (PW 8, CTAS 1): its stage is twice as large
// ([T A_hi atoms][T A_lo atoms][W_hi atom][W_lo atom]), and kSplitWarps more warps (warps 14-17, 576 threads = the launch bound)
// split each landed stage: they wait on full[slot], write hi in place and lo into the lo atom at the same swizzled offset, fence
// the generic-proxy stores against the tensor core's reads and arrive on split[slot], which the MMA warp waits on.  Separate
// warps rather than the producers: the producers never wait for their own copies (cp.async.mbarrier.arrive.noinc), and that is
// what keeps their gathers in flight; a producer that split its rows would have to drain them first.
template <int OP, int PW, int G, int CTAS, bool DET>
__global__ void __launch_bounds__(CTAS == 1 ? 576 : (PW == 8 ? 448 : (SCN_EPI_COLS == 16 ? 384 : 320)), CTAS) conv_plan_tc(const TcParams P) {
  constexpr bool BF16 = OP == kOpBF16 || OP == kOpF16, X3 = OP == kOpTF32X3; // (BF16: 16-bit operands, kind::f16)
  static_assert(!X3 || (PW == 8 && G == 1 && CTAS == 1), "TF32X3: one-CTA configuration only");
  constexpr int TM = G == 4 ? 2 : kMaxT; // tiles per item the producers keep neighbour ids for (G ids per row and tile)
  constexpr int kProdWarps = PW;
  constexpr int kRowsPerWarp = kTileM / PW; // rows of a tile one producer warp gathers
  constexpr int kTakers = 4 + kProdWarps + 1 + (X3 ? kSplitWarps : 0); // warps that take work items from the schedule ring
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nWork = P.nSuper * P.kSplit;
  const uint32_t bBytes = (uint32_t)P.Cout * 128u;
  const uint32_t stageBytes = X3 ? 2u * ((uint32_t)P.T * kAtomBytes + bBytes) : (uint32_t)P.T * kAtomBytes + bBytes; // [T A atoms][B atom] (TF32X3: [T A_hi][T A_lo][W_hi][W_lo])
  unsigned char *sStage = smem;
  float *sEpi = reinterpret_cast<float *>(sStage + (size_t)P.S * stageBytes);
  uint64_t *bars = reinterpret_cast<uint64_t *>(sEpi + kEpiBytes / 4);
  uint64_t *full = bars, *empty = bars + P.S, *accFull = bars + 2 * P.S, *accEmpty = accFull + 2;
  uint32_t *tmemSlot = reinterpret_cast<uint32_t *>(accEmpty + 2);
  uint64_t *split = accEmpty + 3; // TF32X3: [S] stage split into hi / lo (after the TMEM slot word)
  Sched SC{bars + 24, bars + 24 + kSchedSlots, reinterpret_cast<volatile int *>(bars + 24 + 2 * kSchedSlots)}; // (64 barrier words are reserved; 2 S + 5 <= 17 are used above, 3 S + 5 <= 23 with TF32X3)
  const bool dyn = P.sched != nullptr;

  if (tid == 0) {
    for (int i = 0; i < P.S; i++) { mbar_init(smem_u32(full + i), kProdWarps * 32 + 1); mbar_init(smem_u32(empty + i), 1); }
    if constexpr (X3) for (int i = 0; i < P.S; i++) mbar_init(smem_u32(split + i), kSplitWarps * 32);
    for (int i = 0; i < 2; i++) { mbar_init(smem_u32(accFull + i), 1); mbar_init(smem_u32(accEmpty + i), 4); }
    for (int i = 0; i < kSchedSlots; i++) { mbar_init(smem_u32(SC.full + i), 1); mbar_init(smem_u32(SC.empty + i), kTakers); } // takers: epilogue + producer warps + MMA warp (+ split warps; the loader keeps its own copy)
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr int kMmaWarp = 4 + PW;
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmemSlot)), "r"((uint32_t)P.tmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait(); // barriers and TMEM are set up: from here on the kernel reads what the previous kernel on the stream wrote
  const uint32_t tmemBase = *tmemSlot;
  const int accCols = P.T * P.Cout; // columns of one accumulator stage
  const bool prof = P.prof != nullptr;
  long long pw0 = 0, pw1 = 0, pw2 = 0, pw3 = 0;
  const long long tStart = prof ? clock64() : 0;

  if (warp < 4) {
    // ============================ epilogue ============================
    // warp w owns TMEM lanes 32w.. = rows 32w.. of every tile.  Per 32-column block: tcgen05.ld ->
    // padded shared-memory block -> each store instruction writes four whole 128-byte row segments.
    // EC = columns per round (kEpiCols): EC / 4 lanes cover one EC*4-byte row segment, 128 / EC rows per instruction.
    constexpr int EC = kEpiCols, LPR = EC / 4, RPI = 32 / LPR, NI = 32 / RPI; // lanes per row, rows per instruction, instructions per 32 rows
    float *stg = sEpi + warp * (32 * EC);
    const int cl = lane % LPR, cc = cl * 4, rsub = lane / LPR;
    float4 sAcc = make_float4(0.f, 0.f, 0.f, 0.f), qAcc = sAcc; // column sums of the EC-column block this lane group owns (block == rsub)
    for (int it = 0;; it++) {
      const int wi = dyn ? sched_take(SC, it, lane == 0) : (int)(blockIdx.x + (long)it * gridDim.x < nWork ? blockIdx.x + it * gridDim.x : -1);
      if (wi < 0) break;
      const Item I = load_item<G>(P, wi);
      const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
      int myRow[kMaxT]; // output row of (tile t, TMEM lane), fetched before the accumulators are ready
#pragma unroll
      for (int t = 0; t < kMaxT; t++) {
        const long p = (long)(I.st * P.T + t) * kTileM + warp * 32 + lane;
        myRow[t] = (t < P.T && p < P.nOut) ? (P.outRow ? __ldg(P.outRow + p) : (int)p) : -1;
      }
      mbar_wait_t(smem_u32(accFull + a), use & 1, pw0, prof);
      tc_fence_after();
#pragma unroll
      for (int t = 0; t < kMaxT; t++) {
        if (t >= P.T || I.st * P.T + t >= P.nTiles) continue;
        const bool started = I.m[t] != 0ull;
        if (!started && P.kSplit > 1 && !(DET && P.part) && !((P.addend || P.bias) && I.part == 0)) continue; // nothing to add (a partial slot is written even then)
        int rows[NI];
#pragma unroll
        for (int i = 0; i < NI; i++) rows[i] = __shfl_sync(0xffffffffu, myRow[t], i * RPI + rsub);
        for (int c0 = 0; c0 < P.Cout; c0 += EC) {
          uint32_t v[EC];
          if (started) {
            const uint32_t taddr = tmemBase + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * accCols + t * P.Cout + c0);
            tmem_ld(taddr, v); // .x32 or .x16 by the array size
          } else {
#pragma unroll
            for (int j = 0; j < EC; j++) v[j] = 0u;
          }
          __syncwarp();
          // 16-byte chunk q of row r is stored at chunk position q ^ sw(r); sw keeps both the row-wise writes and the
          // column-wise reads free of bank conflicts (EC = 32: r & 7; EC = 16: (r >> 1) & 3, two rows per 128 bytes)
#pragma unroll
          for (int j = 0; j < EC; j += 4)
            *reinterpret_cast<float4 *>(stg + lane * EC + ((((j >> 2) ^ (EC == 32 ? (lane & 7) : ((lane >> 1) & 3)))) << 2)) =
                make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          __syncwarp();
          float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (P.bias && I.part == 0) bv = __ldg(reinterpret_cast<const float4 *>(P.bias + c0 + cc));
          float4 o[NI];
#pragma unroll
          for (int i = 0; i < NI; i++) {
            const int r = i * RPI + rsub;
            o[i] = *reinterpret_cast<const float4 *>(stg + r * EC + ((cl ^ (EC == 32 ? (r & 7) : ((r >> 1) & 3))) << 2));
            o[i].x += bv.x; o[i].y += bv.y; o[i].z += bv.z; o[i].w += bv.w;
          }
          if (P.addend && I.part == 0) {
#pragma unroll
            for (int h = 0; h < NI; h += 4) { // four 16-byte loads in flight per thread
              float4 ad[4];
#pragma unroll
              for (int i = 0; i < 4; i++)
                ad[i] = rows[h + i] >= 0 ? __ldg(reinterpret_cast<const float4 *>(P.addend + (size_t)rows[h + i] * P.ldo + c0 + cc)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
              for (int i = 0; i < 4; i++) { o[h + i].x += ad[i].x; o[h + i].y += ad[i].y; o[h + i].z += ad[i].z; o[h + i].w += ad[i].w; }
            }
          }
          if (P.stats) { // launcher guarantees kSplit == 1 and Cout <= 128: o[] holds final output values
            float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), q4 = s4;
#pragma unroll
            for (int i = 0; i < NI; i++)
              if (rows[i] >= 0) {
                s4.x += o[i].x; s4.y += o[i].y; s4.z += o[i].z; s4.w += o[i].w;
                q4.x = fmaf(o[i].x, o[i].x, q4.x); q4.y = fmaf(o[i].y, o[i].y, q4.y); q4.z = fmaf(o[i].z, o[i].z, q4.z); q4.w = fmaf(o[i].w, o[i].w, q4.w);
              }
#pragma unroll
            for (int d = LPR; d <= 16; d <<= 1) { // the RPI lanes that hold the same columns
              s4.x += __shfl_xor_sync(0xffffffffu, s4.x, d); s4.y += __shfl_xor_sync(0xffffffffu, s4.y, d);
              s4.z += __shfl_xor_sync(0xffffffffu, s4.z, d); s4.w += __shfl_xor_sync(0xffffffffu, s4.w, d);
              q4.x += __shfl_xor_sync(0xffffffffu, q4.x, d); q4.y += __shfl_xor_sync(0xffffffffu, q4.y, d);
              q4.z += __shfl_xor_sync(0xffffffffu, q4.z, d); q4.w += __shfl_xor_sync(0xffffffffu, q4.w, d);
            }
            if (rsub == c0 / EC) { // Cout / EC <= RPI blocks, one per lane group
              sAcc.x += s4.x; sAcc.y += s4.y; sAcc.z += s4.z; sAcc.w += s4.w;
              qAcc.x += q4.x; qAcc.y += q4.y; qAcc.z += q4.z; qAcc.w += q4.w;
            }
          }
          if (P.kSplit == 1) {
#pragma unroll
            for (int i = 0; i < NI; i++)
              if (rows[i] >= 0) {
                if (P.out) *reinterpret_cast<float4 *>(P.out + (size_t)rows[i] * P.ldo + c0 + cc) = o[i]; // null: only the bf16 copy is consumed
                if (P.out16) {
                  uint2 *dst16 = reinterpret_cast<uint2 *>(static_cast<unsigned char *>(P.out16) + ((size_t)rows[i] * P.ldo + c0 + cc) * 2);
                  if (OP == kOpF16 || (OP == kOpTF32 && P.f16)) *dst16 = pack16x4<true>(o[i]);
                  else *dst16 = pack16x4<false>(o[i]);
                }
              }
          } else if (DET && P.part) { // offsets split over CTAs, deterministic mode: this split's partial rows into its own slot
#pragma unroll
            for (int i = 0; i < NI; i++)
              if (rows[i] >= 0) *reinterpret_cast<float4 *>(P.part + ((size_t)I.part * P.nOut + rows[i]) * P.Cout + c0 + cc) = o[i];
          } else { // offsets split over CTAs: accumulate into the launcher-zeroed output
#pragma unroll
            for (int i = 0; i < NI; i++)
              if (rows[i] >= 0) {
                float *dst = P.out + (size_t)rows[i] * P.ldo + c0 + cc;
                atomicAdd(dst, o[i].x); atomicAdd(dst + 1, o[i].y); atomicAdd(dst + 2, o[i].z); atomicAdd(dst + 3, o[i].w);
              }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(accEmpty + a));
      if (DET && P.statsPart) { // deterministic mode: this item's sums of this warp's rows into slot (item, warp); the launcher adds the slots in order
        const int c = rsub * EC + cc;
        if (c < P.Cout) {
          double *dst = P.statsPart + ((size_t)wi * 4 + warp) * 2 * P.Cout + c;
          dst[0] = sAcc.x; dst[1] = sAcc.y; dst[2] = sAcc.z; dst[3] = sAcc.w;
          dst += P.Cout;
          dst[0] = qAcc.x; dst[1] = qAcc.y; dst[2] = qAcc.z; dst[3] = qAcc.w;
        }
        sAcc = make_float4(0.f, 0.f, 0.f, 0.f);
        qAcc = sAcc;
      }
    }
    if (P.stats && !(DET && P.statsPart)) { // one double atomic per (warp, channel) into one of kBnReplicas accumulators
      const int c = rsub * EC + cc;
      if (c < P.Cout) {
        double *rep = P.stats + (size_t)(blockIdx.x % kBnReplicas) * 2 * kFusedStatsC;
        atomicAdd(rep + c, (double)sAcc.x); atomicAdd(rep + c + 1, (double)sAcc.y); atomicAdd(rep + c + 2, (double)sAcc.z); atomicAdd(rep + c + 3, (double)sAcc.w);
        rep += kFusedStatsC;
        atomicAdd(rep + c, (double)qAcc.x); atomicAdd(rep + c + 1, (double)qAcc.y); atomicAdd(rep + c + 2, (double)qAcc.z); atomicAdd(rep + c + 3, (double)qAcc.w);
      }
    }
    if (prof && tid == 0) { P.prof[blockIdx.x * 32 + 0] = clock64() - tStart; P.prof[blockIdx.x * 32 + 1] = pw0; }
  } else if (warp < 4 + kProdWarps) {
    // ============================ A producers ============================
    // Warp pw gathers rows [R pw, R pw + R) of every tile of the stage (R = 128 / PW): R / 4 cp.async
    // instructions per tile (8 lanes x 16 B = one 128-byte row chunk, 4 rows per instruction).  The
    // ids of the current filter offset sit in registers (lane l holds row R pw + l % R of each tile)
    // and those of the next active offset are fetched while the current one is gathered.
    const int pw = warp - 4;
    const int chunk = lane & 7, rsub = lane >> 3;
    uint32_t n = 0, slot = 0, round = 0; // stage counter, ring slot, ring round
    for (int itp = 0;; itp++) {
      const int wi = dyn ? sched_take(SC, itp, lane == 0) : (int)(blockIdx.x + (long)itp * gridDim.x < nWork ? blockIdx.x + itp * gridDim.x : -1);
      if (wi < 0) break;
      const Item I = load_item<G>(P, wi);
      if (!I.uni) continue;
      const int *idBase = P.nbr + ((size_t)I.st * P.T * P.K) * 128 + pw * kRowsPerWarp + (lane & (kRowsPerWarp - 1));
      int idc[G][TM], idn[G][TM];
      auto load_ids = [&](int k, int (&dst)[G][TM]) {
#pragma unroll
        for (int g = 0; g < G; g++)
#pragma unroll
          for (int t = 0; t < TM; t++) {
            if (G == 1 && is_lateral(P, k)) { // lateral stage: the input row of an output site is its own output row
              const long p = (long)(I.st * P.T + t) * kTileM + pw * kRowsPerWarp + (lane & (kRowsPerWarp - 1));
              dst[g][t] = (((I.m[t] >> k) & 1ull) && p < P.nOut) ? (P.outRow ? __ldg(P.outRow + p) : (int)p) : -1;
            } else if (!P.nbr) { // dense rows: site p reads row p
              const long p = (long)(I.st * P.T + t) * kTileM + pw * kRowsPerWarp + (lane & (kRowsPerWarp - 1));
              dst[g][t] = (((I.m[t] >> k) & 1ull) && g == 0 && p < P.nOut) ? (int)p : -1;
            } else {
              dst[g][t] = (((I.m[t] >> k) & 1ull) && k + g < P.K) ? __ldg(idBase + ((size_t)t * P.K + k + g) * 128) : -1;
            }
          }
      };
      // packed rows: 16-byte chunk `chunk` of the 128-byte atom row belongs to offset k + myG, bytes [16 sub, 16 sub + 16) of that neighbour's row
      constexpr int kChunksPerRow = 8 / G;
      const int myG = chunk / kChunksPerRow, sub = chunk % kChunksPerRow;
      int k = __ffsll((long long)I.uni) - 1;
      load_ids(k, idn);
      while (k >= 0) {
#pragma unroll
        for (int g = 0; g < G; g++)
#pragma unroll
          for (int t = 0; t < TM; t++) idc[g][t] = idn[g][t];
        const unsigned long long rest = (k + 1 < 64) ? (I.uni >> (k + 1)) : 0ull;
        const int kNext = rest ? k + 1 + (__ffsll((long long)rest) - 1) : -1;
        if (kNext >= 0) load_ids(kNext, idn);
        const bool lat = G == 1 && is_lateral(P, k);
        const unsigned char *srcBase = lat ? P.in2 : P.in;
        const int srcRowBytes = lat ? P.rowBytes2 : P.rowBytes, nA = lat ? P.nAtoms2 : P.nAtoms;
        for (int c = 0; c < nA; c++) {
          n++;
          mbar_wait_t(smem_u32(empty + slot), (round & 1u) ^ 1u, pw0, prof);
          const uint32_t sbase = smem_u32(sStage) + slot * stageBytes;
          // Everything that does not depend on the row is computed once per stage: the producers are paced by their instruction issue
          // rate (ncu: ~20 SASS instructions per copy, waiting for a free slot only a third of the time), so a copy is SHFL + clamp +
          // compare + one IMAD.WIDE (row id x row bytes + per-lane base) + the request.  A missing neighbour (id < 0) or a chunk
          // beyond a narrow row (a 32-channel lateral) requests 0 bytes = zero fill; its address stays inside row 0.
          const bool inRow = G > 1 || c * 128 + chunk * 16 < srcRowBytes;
          unsigned long long laneBase = reinterpret_cast<unsigned long long>(G == 1 ? srcBase + (inRow ? c * 128 + chunk * 16 : 0) : P.in + sub * 16);
          asm volatile("" : "+l"(laneBase)); // one 64-bit value: the address of a row is then a single IMAD.WIDE
          const int notInRow = inRow ? 0 : (int)0x80000000; // OR-ed into the id: such a lane always requests 0 bytes
          const unsigned rowStep = G == 1 ? (unsigned)srcRowBytes : (unsigned)(128 / G);
          const uint32_t dstLane = sbase + (uint32_t)(pw * kRowsPerWarp + rsub) * 128u;
          const uint32_t swz0 = (uint32_t)(chunk ^ rsub) << 4, swz1 = (uint32_t)(chunk ^ (rsub + 4)) << 4; // row & 7 = rsub (i even) or rsub + 4 (i odd)
          if (!(P.dbg & 1)) {
#pragma unroll
            for (int t = 0; t < TM; t++) {
              if (!((I.m[t] >> k) & 1ull)) continue; // uniform over the CTA
#pragma unroll
              for (int i = 0; i < kRowsPerWarp / 4; i++) {
                int id = __shfl_sync(0xffffffffu, idc[0][t], i * 4 + rsub);
#pragma unroll
                for (int g = 1; g < G; g++) {
                  const int v = __shfl_sync(0xffffffffu, idc[g][t], i * 4 + rsub);
                  if (g == myG) id = v;
                }
                id |= notInRow;
                const void *src = reinterpret_cast<const void *>(laneBase + (unsigned long long)(unsigned)max(id, 0) * rowStep);
                cp_async16(dstLane + (uint32_t)(t * kAtomBytes + i * 512) + ((i & 1) ? swz1 : swz0), src, id >= 0 ? 16u : 0u);
              }
            }
          }
          // The stage's full barrier receives this thread's arrival when its copies above have landed
          // (cp.async.mbarrier.arrive.noinc): no wait_group, no fence, the warp moves on to the next free
          // slot at once.  Same hand-off as CUTLASS's sm100 cp.async -> UMMA mainloop
          // (sm100_mma_cpasync_warpspecialized.hpp), which issues tcgen05.mma right after the barrier wait.
          // Measured before: a warp that waited (cp.async.wait_group + fence.proxy.async, i.e. MEMBAR.ALL.CTA)
          // drained ALL its copies at every stage, so deeper rings bought nothing.
          cp_async_mbar_arrive_noinc(smem_u32(full + slot));
          if (++slot == (uint32_t)P.S) { slot = 0; round++; }
        }
        k = kNext;
      }
    }
    if (prof && lane == 0 && pw == 0) { long long *q = P.prof + blockIdx.x * 32 + 4; q[0] = clock64() - tStart; q[1] = pw0; q[2] = pw1; q[3] = n; }
  } else if (warp == kMmaWarp) {
    // ============================ MMA issuer ============================
    // The whole warp runs the control flow (converged), one elected lane issues: ptxas then keeps
    // descriptors in uniform registers and emits straight-line UTCHMMA instead of a per-instruction
    // election loop (measured: ~120 cycles per MMA issued from a divergent `if (lane == 0)` region).
    {
      // instruction descriptor: D=F32, A/B = TF32 (2), BF16 (1) or F16 (0), K-major both, N=Cout, M=128
      const uint32_t fmt = OP == kOpF16 ? 0u : BF16 ? 1u : 2u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(P.Cout >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
      uint32_t n = 0, slot = 0, round = 0;
      const uint32_t sStage0 = smem_u32(sStage), full0 = smem_u32(full), empty0 = smem_u32(empty);
      for (int it = 0;; it++) {
        const int wi = dyn ? sched_take(SC, it, lane == 0) : (int)(blockIdx.x + (long)it * gridDim.x < nWork ? blockIdx.x + it * gridDim.x : -1);
        if (wi < 0) break;
        const Item I = load_item<G>(P, wi);
        const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
        mbar_wait_t(smem_u32(accEmpty + a), (use & 1) ^ 1, pw0, prof); // epilogue has drained this accumulator stage
        tc_fence_after();
        uint32_t started = 0;
        unsigned long long rest = I.uni;
        while (rest) {
          const int k = __ffsll((long long)rest) - 1;
          rest &= rest - 1;
          const int nA = (G == 1 && is_lateral(P, k)) ? P.nAtoms2 : P.nAtoms;
          for (int c = 0; c < nA; c++) {
            n++;
            mbar_wait_t(full0 + slot * 8u, round & 1u, pw1, prof);
            if constexpr (X3) mbar_wait_t(smem_u32(split + slot), round & 1u, pw1, prof); // (full: the weight atoms; split: the A atoms, split and fenced)
            tc_fence_after();
            const uint32_t sbase = sStage0 + slot * stageBytes;
            const uint64_t bDesc = smem_desc_sw128(sbase + (X3 ? 2u * (uint32_t)P.T * kAtomBytes : (uint32_t)P.T * kAtomBytes));
            const long long tI0 = prof ? clock64() : 0;
            if (elect_one()) {
              if (!(P.dbg & 4)) {
#pragma unroll
                for (int t = 0; t < kMaxT; t++) {
                  if (!((I.m[t] >> k) & 1ull)) continue;
                  const uint64_t aDesc = smem_desc_sw128(sbase + t * kAtomBytes);
                  const uint32_t d = tmemBase + (uint32_t)(a * accCols + t * P.Cout);
                  if constexpr (X3) {
                    const uint64_t aLoDesc = smem_desc_sw128(sbase + (uint32_t)(P.T + t) * kAtomBytes), bLoDesc = smem_desc_sw128(sbase + 2u * (uint32_t)P.T * kAtomBytes + bBytes);
#pragma unroll
                    for (int j = 0; j < 4; j++) { // per 32 bytes of K: the two small terms first, then A_hi W_hi
                      tc_mma<false>(d, aDesc + (uint64_t)(j * 2), bLoDesc + (uint64_t)(j * 2), idesc, ((started >> t) & 1u) | (j > 0));
                      tc_mma<false>(d, aLoDesc + (uint64_t)(j * 2), bDesc + (uint64_t)(j * 2), idesc, 1u);
                      tc_mma<false>(d, aDesc + (uint64_t)(j * 2), bDesc + (uint64_t)(j * 2), idesc, 1u);
                    }
                  } else {
#pragma unroll
                    for (int j = 0; j < 4; j++) // 4 x 32 bytes of K inside the 128-byte swizzle atom
                      tc_mma<BF16>(d, aDesc + (uint64_t)(j * 2), bDesc + (uint64_t)(j * 2), idesc, ((started >> t) & 1u) | (j > 0));
                  }
                }
              }
              const long long tI1 = prof ? clock64() : 0;
              tc_commit(empty0 + slot * 8u);
              if (prof) { pw2 += tI1 - tI0; pw3 += clock64() - tI1; }
            }
            __syncwarp();
#pragma unroll
            for (int t = 0; t < kMaxT; t++) started |= (uint32_t)((I.m[t] >> k) & 1ull) << t;
            if (++slot == (uint32_t)P.S) { slot = 0; round++; }
          }
        }
        if (elect_one()) tc_commit(smem_u32(accFull + a));
        __syncwarp();
      }
      if (prof) { // pw2/pw3 live in whichever lane was elected
        long long *q = P.prof + blockIdx.x * 32 + 10;
        if (lane == 0) { q[0] = clock64() - tStart; q[1] = pw0; q[2] = pw1; q[3] = n; }
        if (pw2 | pw3) { q[4] = pw2; q[5] = pw3; }
      }
    }
  } else if (!X3 || warp == kMmaWarp + 1) {
    // ============================ B loader ============================
    if (lane == 0) {
      uint32_t n = 0, slot = 0, round = 0;
      // this thread also draws the work items (dynamic distribution): item itb is published before it is used here, item itb + 1
      // is drawn while item itb is being loaded
      int cur = 0, nxt = -1;
      if (dyn) { cur = sched_draw(P, nWork); sched_publish(SC, 0, cur); nxt = cur >= 0 ? sched_draw(P, nWork) : -1; }
      for (int itb = 0;; itb++) {
        int wi;
        if (dyn) {
          if (cur < 0) break;
          sched_publish(SC, itb + 1, nxt);
          const int nn = nxt >= 0 ? sched_draw(P, nWork) : -1;
          wi = cur; cur = nxt; nxt = nn;
        } else {
          if (blockIdx.x + (long)itb * gridDim.x >= nWork) break;
          wi = blockIdx.x + itb * gridDim.x;
        }
        const Item I = load_item<G>(P, wi);
        unsigned long long rest = I.uni;
        while (rest) {
          const int k = __ffsll((long long)rest) - 1;
          rest &= rest - 1;
          const bool lat = G == 1 && is_lateral(P, k);
          const int w = lat ? 0 : (P.tileW ? __ldg(P.tileW + I.st) : k / G); // packed: one weight atom per offset group
          const unsigned char *wsrc = lat ? P.wimg2 : P.wimg;
          const int nA = lat ? P.nAtoms2 : P.nAtoms;
          for (int c = 0; c < nA; c++) {
            n++;
            mbar_wait_t(smem_u32(empty + slot), (round & 1u) ^ 1u, pw0, prof);
            const uint32_t bar = smem_u32(full + slot);
            if (P.dbg & 2) { mbar_arrive(bar); }
            else {
              if constexpr (X3) { // the W_hi and W_lo atoms lie side by side in the image and in the stage
                mbar_arrive_expect_tx(bar, 2u * bBytes);
                bulk_g2s(smem_u32(sStage) + slot * stageBytes + 2u * (uint32_t)P.T * kAtomBytes, wsrc + ((size_t)w * nA + c) * 2u * bBytes, 2u * bBytes, bar);
              } else {
                mbar_arrive_expect_tx(bar, bBytes);
                bulk_g2s(smem_u32(sStage) + slot * stageBytes + (uint32_t)P.T * kAtomBytes, wsrc + ((size_t)w * nA + c) * bBytes, bBytes, bar);
              }
            }
            if (++slot == (uint32_t)P.S) { slot = 0; round++; }
          }
        }
      }
      if (prof) { long long *q = P.prof + blockIdx.x * 32 + 16; q[0] = clock64() - tStart; q[1] = pw0; q[2] = n; }
    }
  } else if constexpr (X3) {
    // ============================ operand split (TF32X3) ============================
    // The 128 threads walk the stages in the MMA warp's order; of every live tile each thread rewrites 8 of the 1024 16-byte
    // chunks (consecutive threads, consecutive chunks: conflict-free): hi = tf32(x) in place, lo = tf32(x - hi) at the same
    // offset of the lo atom (the 128-byte swizzle depends on the offset within the 1024-aligned atom only, so the lo atom
    // needs no swizzle of its own).  Zero-filled rows (no neighbour) split into zeros.
    const int st = tid - (kMmaWarp + 2) * 32;
    uint32_t slot = 0, round = 0;
    const uint32_t full0 = smem_u32(full), split0 = smem_u32(split);
    for (int it = 0;; it++) {
      const int wi = dyn ? sched_take(SC, it, lane == 0) : (int)(blockIdx.x + (long)it * gridDim.x < nWork ? blockIdx.x + it * gridDim.x : -1);
      if (wi < 0) break;
      const Item I = load_item<G>(P, wi);
      unsigned long long rest = I.uni;
      while (rest) {
        const int k = __ffsll((long long)rest) - 1;
        rest &= rest - 1;
        const int nA = (G == 1 && is_lateral(P, k)) ? P.nAtoms2 : P.nAtoms;
        for (int c = 0; c < nA; c++) {
          mbar_wait(full0 + slot * 8u, round & 1u);
          unsigned char *sb = sStage + (size_t)slot * stageBytes;
#pragma unroll
          for (int t = 0; t < kMaxT; t++) {
            if (!((I.m[t] >> k) & 1ull)) continue;
            float4 *hi = reinterpret_cast<float4 *>(sb + t * kAtomBytes), *lo = reinterpret_cast<float4 *>(sb + (size_t)(P.T + t) * kAtomBytes);
#pragma unroll
            for (int i = 0; i < kAtomBytes / 16 / (kSplitWarps * 32); i++) {
              const int q = i * kSplitWarps * 32 + st;
              const float4 x = hi[q];
              float4 h, l;
              tf32_split(x.x, h.x, l.x); tf32_split(x.y, h.y, l.y); tf32_split(x.z, h.z, l.z); tf32_split(x.w, h.w, l.w);
              hi[q] = h;
              lo[q] = l;
            }
          }
          fence_proxy_async(); // generic-proxy stores -> the tensor core's (async proxy) reads
          mbar_arrive(split0 + slot * 8u);
          if (++slot == (uint32_t)P.S) { slot = 0; round++; }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"((uint32_t)P.tmemCols) : "memory");
  }
}

// W [K][Cin][Cout] fp32 -> per (k, 128-byte K atom) the exact shared-memory image of the B operand:
// Cout rows x 128 bytes (32 tf32 / 64 bf16 input channels of one output channel), 16-byte chunks
// XOR-swizzled by (row & 7); values rounded to nearest (TF32: cvt.rna, BF16 / F16: rn, fp16 overflowing to +-inf).
// Cin = padded channel count of the image (multiple of the atom width), CinW = channels W really has.
// wT: 0 = W is [K][CinW][Cout]; 1 / 2 = the operand is the TRANSPOSE of a forward weight tensor stored as [K][Cout][CinW] (the input-gradient
// convolutions: Wt[k'][co][ci] = W[k][ci][co]), 2 = with the filter offsets reversed as well (k' = K - 1 - k) -- read in place, no transposed copy.
// el = element format: 0 = tf32, kWimgBF16, kWimgF16.
// co0, ldW: the image holds output channels [co0, co0 + Cout) of a W whose output dimension is ldW wide (a column slab; 0, Cout otherwise).
__global__ void k_prep_wimg(const float *__restrict__ W, unsigned char *__restrict__ img, int K, int Cin, int CinW, int Cout, int el, int wT, int co0, int ldW) {
  const bool bf16 = el != 0; // (2-byte elements)
  const long n = (long)K * Cin * Cout;
  const int per = bf16 ? 64 : 32, nAtoms = Cin / per;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const long t = i / Cout;
    const int ci = (int)(t % Cin), k = (int)(t / Cin);
    const int c = ci / per, j = ci % per;
    const int byte = j * (bf16 ? 2 : 4), chunk = byte >> 4, within = byte & 15;
    unsigned char *dst = img + ((long)k * nAtoms + c) * Cout * 128 + (long)co * 128 + ((chunk ^ (co & 7)) << 4) + within;
    const int ks = wT == 2 ? K - 1 - k : k;
    const float w = ci < CinW ? (wT ? W[((long)ks * ldW + co0 + co) * CinW + ci] : W[((long)k * CinW + ci) * ldW + co0 + co]) : 0.f;
    if (el == 3) { // (kWimgF16)
      *reinterpret_cast<unsigned short *>(dst) = to16<true>(w);
    } else if (bf16) {
      *reinterpret_cast<unsigned short *>(dst) = to16<false>(w);
    } else {
      uint32_t r;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(w));
      *reinterpret_cast<uint32_t *>(dst) = r;
    }
  }
}

// TF32X3 operands: the same image twice per (k, K atom), [W_hi atom][W_lo atom] side by side (one bulk copy per stage),
// W_hi = tf32(w) and W_lo = tf32(w - W_hi), both exact TF32 values.  Same arguments as k_prep_wimg.
__global__ void k_prep_wimg_split(const float *__restrict__ W, unsigned char *__restrict__ img, int K, int Cin, int CinW, int Cout, int wT, int co0, int ldW) {
  const long n = (long)K * Cin * Cout;
  const int nAtoms = Cin / 32;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const long t = i / Cout;
    const int ci = (int)(t % Cin), k = (int)(t / Cin);
    const int c = ci / 32, j = ci % 32;
    const int byte = j * 4, chunk = byte >> 4, within = byte & 15;
    unsigned char *dst = img + ((long)k * nAtoms + c) * 2 * Cout * 128 + (long)co * 128 + ((chunk ^ (co & 7)) << 4) + within;
    const int ks = wT == 2 ? K - 1 - k : k;
    const float w = ci < CinW ? (wT ? W[((long)ks * ldW + co0 + co) * CinW + ci] : W[((long)k * CinW + ci) * ldW + co0 + co]) : 0.f;
    float hi, lo;
    tf32_split(w, hi, lo);
    *reinterpret_cast<float *>(dst) = hi;
    *reinterpret_cast<float *>(dst + (long)Cout * 128) = lo;
  }
}

// Packed layers (16-bit rows of 128 / G bytes, G = 2 or 4; fp16 elements with f16, else bf16): the K atom of offset group kg holds, for output channel co,
// [offset kg G | offset kg G + 1 | ...] x Cin input channels -- the same order in which the producers lay the G
// gathered neighbour rows side by side.  Offsets beyond K and channels beyond CinW are zero.
__global__ void k_prep_wimg_packed(const float *__restrict__ W, unsigned char *__restrict__ img, int K, int G, int Cin, int CinW, int Cout, int wT, int f16, int co0,
                                   int ldW) {
  const int KG = (K + G - 1) / G;
  const long n = (long)KG * G * Cin * Cout;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const long t = i / Cout;
    const int ci = (int)(t % Cin), k = (int)(t / Cin);
    const int kg = k / G, g = k % G;
    const int byte = (g * Cin + ci) * 2, chunk = byte >> 4, within = byte & 15;
    unsigned char *dst = img + (long)kg * Cout * 128 + (long)co * 128 + ((chunk ^ (co & 7)) << 4) + within;
    const int ks = wT == 2 ? K - 1 - k : k;
    const float w = (k < K && ci < CinW) ? (wT ? W[((long)ks * ldW + co0 + co) * CinW + ci] : W[((long)k * CinW + ci) * ldW + co0 + co]) : 0.f;
    *reinterpret_cast<unsigned short *>(dst) = f16 ? to16<true>(w) : to16<false>(w);
  }
}

// Weight images are cached across calls: (device pointer, caller's version tag, shape, operand
// type) -> image.  The tag is how the caller says "same contents as last time" (the Python layer
// passes a per-Parameter token combined with the tensor's in-place version counter); tag 0 = no caching.
struct WimgKey {
  const void *w; long long tag; int K, Cin, CinW, Cout, fmt, dev; // fmt: element format and packing of the image (launch_prep_wimg)
  int co0, ldW;                                                   // the output columns of a slab (k_prep_wimg): one image per slab
  bool operator<(const WimgKey &o) const {
    return std::tie(w, tag, K, Cin, CinW, Cout, fmt, dev, co0, ldW) < std::tie(o.w, o.tag, o.K, o.Cin, o.CinW, o.Cout, o.fmt, o.dev, o.co0, o.ldW);
  }
};
struct WimgVal { unsigned char *img; size_t bytes; cudaEvent_t ready; cudaStream_t stream; unsigned long long lastUse; };
static std::map<WimgKey, WimgVal> g_wimg;
static std::mutex g_wimg_mu;
static size_t g_wimg_bytes = 0;
static unsigned long long g_wimg_clock = 0;
constexpr size_t kWimgBudget = 768u << 20;
// Returns the image; *owned = true when the caller must cudaFreeAsync it (uncached).
// fmt: element format (0 = tf32, kWimgBF16, kWimgSplit = tf32 hi / lo pairs (TF32X3), kWimgF16) + 16 G for packed 16-bit images (G
// offsets per atom).  The format is part of the cache key: the images of one weight tensor in different modes -- bf16 and fp16
// included -- are separate entries, so a mode switch never hands a kernel an image in the other format.
constexpr int kWimgBF16 = 1, kWimgSplit = 2, kWimgF16 = 3;
static void launch_prep_wimg(const float *W, unsigned char *img, int K, int Cin, int CinW, int Cout, int fmt, cudaStream_t s, int wT, int co0, int ldW) {
  const int G = fmt >> 4;
  if (G > 1) k_prep_wimg_packed<<<stream_grid((long)((K + G - 1) / G) * G * Cin * Cout, 256), 256, 0, LS(s)>>>(W, img, K, G, Cin, CinW, Cout, wT, (fmt & 15) == kWimgF16, co0, ldW);
  else if (fmt == kWimgSplit) k_prep_wimg_split<<<stream_grid((long)K * Cin * Cout, 256), 256, 0, LS(s)>>>(W, img, K, Cin, CinW, Cout, wT, co0, ldW);
  else k_prep_wimg<<<stream_grid((long)K * Cin * Cout, 256), 256, 0, LS(s)>>>(W, img, K, Cin, CinW, Cout, fmt & 15, wT, co0, ldW);
}
// co0, ldW: output columns [co0, co0 + Cout) of a W ldW wide (a column slab); ldW = 0: Cout
static int get_wimg(const float *W, long long tag, int K, int Cin, int CinW, int Cout, int fmt, cudaStream_t s, unsigned char **img, bool *owned, int wT = 0,
                    int co0 = 0, int ldW = 0) {
  if (!ldW) ldW = Cout;
  if (wT) tag = 0; // (transposed operands belong to the backward pass of a training step: the weights change every step, nothing to cache)
  const int packG = fmt >> 4;
  const size_t bytes = packG > 1 ? (size_t)((K + packG - 1) / packG) * Cout * 128 : (size_t)K * Cin * Cout * (fmt == kWimgSplit ? 8 : fmt ? 2 : 4);
  *owned = false;
  if (tag != 0) {
    int dev = 0;
    SCN_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_wimg_mu);
    WimgKey key{W, tag, K, Cin, CinW, Cout, fmt, dev, co0, ldW};
    auto it = g_wimg.find(key);
    if (it != g_wimg.end()) {
      it->second.lastUse = ++g_wimg_clock;
      if (it->second.stream != s) SCN_CUDA(cudaStreamWaitEvent(s, it->second.ready, 0));
      *img = it->second.img;
      return 0;
    }
    // stale versions of the same weight tensor, then least-recently-used entries beyond the budget
    for (auto j = g_wimg.begin(); j != g_wimg.end();) {
      if (j->first.w == W && j->first.dev == dev && j->first.tag != tag) { cudaFree(j->second.img); cudaEventDestroy(j->second.ready); g_wimg_bytes -= j->second.bytes; j = g_wimg.erase(j); }
      else ++j;
    }
    while (g_wimg_bytes + bytes > kWimgBudget && !g_wimg.empty()) {
      auto lru = g_wimg.begin();
      for (auto j = g_wimg.begin(); j != g_wimg.end(); ++j) if (j->second.lastUse < lru->second.lastUse) lru = j;
      cudaFree(lru->second.img); cudaEventDestroy(lru->second.ready); g_wimg_bytes -= lru->second.bytes; g_wimg.erase(lru);
    }
    WimgVal v;
    SCN_CUDA(cudaMalloc((void **)&v.img, bytes));
    SCN_CUDA(cudaEventCreateWithFlags(&v.ready, cudaEventDisableTiming));
    launch_prep_wimg(W, v.img, K, Cin, CinW, Cout, fmt, s, 0, co0, ldW);
    SCN_CUDA(cudaEventRecord(v.ready, s));
    v.bytes = bytes; v.stream = s; v.lastUse = ++g_wimg_clock;
    g_wimg[key] = v;
    g_wimg_bytes += bytes;
    *img = v.img;
    return 0;
  }
  SCN_CUDA(cudaMallocAsync((void **)img, bytes, s));
  launch_prep_wimg(W, *img, K, Cin, CinW, Cout, fmt, s, wT, co0, ldW);
  *owned = true;
  return 0;
}

int tc_available() {
  static int cached = -1;
  if (cached < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) major = 0;
    cached = major == 10;
  }
  return cached;
}

__global__ void k_pad_rows(const float *__restrict__ in, float *__restrict__ out, long n, int C, int Cp) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n * Cp; i += (long)gridDim.x * blockDim.x) {
    int c = (int)(i % Cp);
    out[i] = c < C ? __ldg(in + (i / Cp) * C + c) : 0.f;
  }
}
// rows of C <= Cp channels -> 16-bit rows (bf16, or fp16 with F16) zero-padded to Cp channels (the 9-channel network input -> 16
// channels = 32-byte rows)
template <bool F16>
__global__ void k_pad_rows16(const float *__restrict__ in, unsigned short *__restrict__ out, long n, int C, int Cp) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n * Cp; i += (long)gridDim.x * blockDim.x) {
    int c = (int)(i % Cp);
    out[i] = to16<F16>(c < C ? __ldg(in + (i / Cp) * C + c) : 0.f);
  }
}
static void launch_pad_rows16(const float *in, void *out, long n, int C, int Cp, bool f16, cudaStream_t s) {
  if (f16) k_pad_rows16<true><<<stream_grid(n * Cp, 256), 256, 0, LS(s)>>>(in, static_cast<unsigned short *>(out), n, C, Cp);
  else k_pad_rows16<false><<<stream_grid(n * Cp, 256), 256, 0, LS(s)>>>(in, static_cast<unsigned short *>(out), n, C, Cp);
}
// fp32 -> 16-bit (rn) copy of a feature matrix (bf16, or fp16 with F16), for inputs that arrive without a 16-bit shadow
template <bool F16>
__global__ void __launch_bounds__(256) k_to_16(const float *__restrict__ x, uint2 *__restrict__ y, long n4) {
  pdl_launch_dependents();
  pdl_wait();
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(x) + i);
    y[i] = pack16x4<F16>(v);
  }
}
static cudaError_t launch_to_16(const float *x, void *y, long n4, bool f16, cudaStream_t s) {
  if (f16) return launch_pdl(k_to_16<true>, dim3(stream_grid(n4, 256)), dim3(256), 0, LS(s), x, static_cast<uint2 *>(y), n4);
  return launch_pdl(k_to_16<false>, dim3(stream_grid(n4, 256)), dim3(256), 0, LS(s), x, static_cast<uint2 *>(y), n4);
}
// the 16-bit copy of x in the current mode's format (common.cuh)
int to_16(const float *x, void *y, long n, cudaStream_t s) {
  SCN_CHECK(n % 4 == 0, "16-bit copy needs an element count that is a multiple of 4");
  if (n) SCN_CUDA(launch_to_16(x, y, n / 4, f16_copies(), s));
  SCN_CUDA(cudaGetLastError());
  return 0;
}
// deterministic mode, split filter offsets: out = partial of split 0 + split 1 + ... in that order (bias and addend are in split 0's),
// with the 16-bit copy of the finished rows (what the memset + atomic epilogue + k_to_16 do otherwise).  The n4 / cols4 rows of cols4
// float4s lie pld4 (part) and ld4 (out, out16) apart -- a column slab of wider rows; part slice k starts at k n4 / cols4 pld4.  With
// part == out and kSplit == 1 (out == null): the 16-bit copy of a slab's finished columns.
template <bool F16>
__global__ void __launch_bounds__(256) k_split_sum(const float4 *__restrict__ part, int kSplit, long n4, int cols4, int pld4, int ld4, float4 *__restrict__ out,
                                                   uint2 *__restrict__ out16) {
  pdl_launch_dependents();
  pdl_wait();
  const long slice = n4 / cols4 * pld4;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const long r = i / cols4, j = i - r * cols4, ip = r * pld4 + j, io = r * ld4 + j;
    float4 a = part[ip];
    for (int k = 1; k < kSplit; k++) {
      const float4 b = part[(long)k * slice + ip];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (out) out[io] = a;
    if (out16) out16[io] = pack16x4<F16>(a);
  }
}
static int stream_scratch(cudaStream_t s, int slot, size_t bytes, void **out);
// 16-bit copy of a backward call's d_out, made once and read by both the input-gradient and the weight-gradient kernel
int dout16_copy(const float *d_out, long n, cudaStream_t s, const void **out) {
  void *p = nullptr;
  SCN_TRY(stream_scratch(s, 3, (size_t)n * 2 + 16, &p));
  SCN_TRY(to_16(d_out, p, n, s));
  *out = p;
  return 0;
}
// Grow-only scratch per (device, stream, slot) for the operand copies a call may need (slot 0: zero-padded rows of a
// narrow input; slot 1: bf16 copy of an input that arrived without one -- one launch can need both, the second derived
// from the first, so they must not share a buffer; slot 2: the operand pair of the weight-gradient kernel).  Uses of a
// slot on one stream are ordered; cudaMallocAsync took milliseconds for these 150-300 MB blocks.
// 3: bf16 copy of d_out shared by the two gradient kernels of a backward call; 4: partial sums of the deterministic mode (det_scratch)
// 5: running sums of a chunked launch (launch_conv_plan_tc_chunked)
enum ScratchSlot { kScratchPad = 0, kScratchBf16 = 1, kScratchDw = 2, kScratchDout = 3, kScratchDet = 4, kScratchChunk = 5 };
static std::mutex g_scratch_mu;
static std::map<std::tuple<int, cudaStream_t, int>, std::pair<void *, size_t>> g_scratch;
static int stream_scratch(cudaStream_t s, int slot, size_t bytes, void **out) {
  int dev = 0;
  SCN_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_scratch_mu);
  auto &e = g_scratch[std::make_tuple(dev, s, slot)];
  if (e.second < bytes) {
    if (e.first) { SCN_CUDA(cudaStreamSynchronize(s)); SCN_CUDA(cudaFree(e.first)); }
    e.second = bytes + bytes / 8 + (1u << 20);
    SCN_CUDA(cudaMalloc(&e.first, e.second));
  }
  *out = e.first;
  return 0;
}
int det_scratch(cudaStream_t s, size_t bytes, void **out) { return stream_scratch(s, kScratchDet, bytes, out); }
// Work-item counters of the dynamic distribution: two zero-initialised words per (device, stream); launches on one stream are
// ordered and every launch leaves them zeroed again (sched_draw).
static int sched_counters(cudaStream_t s, unsigned **out) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, unsigned *> cache;
  int dev = 0;
  SCN_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  unsigned *&e = cache[std::make_pair(dev, s)];
  if (!e) {
    SCN_CUDA(cudaMalloc((void **)&e, 64));
    SCN_CUDA(cudaMemset(e, 0, 64));
  }
  *out = e;
  return 0;
}
// A plan of more than 64 filter offsets (chunk-major, common.cuh) runs as one launch per chunk of <= 63 offsets.  Chunk c is an
// ordinary plan -- its own block of neighbour ids and mask array, the weights of its offsets -- and takes the running sum of the
// chunks before it as its fused addend.  Bias and the caller's addend go into chunk 0; the lateral stage, the epilogue statistics
// and the bf16 copy into the last chunk, the only one that sees finished rows.  The running sums alternate between two scratch
// buffers, so no launch reads rows it writes (an offset-split launch zeroes its output first).  Each chunk boundary adds one fp32
// rounding of the partial sum (DESIGN.md section 7).
static int launch_conv_plan_tc_chunked(const TcConv &c, cudaStream_t s) {
  const int K = c.K, CinW = c.CinW ? c.CinW : c.Cin, nC = plan_chunks(K);
  const long nPad = plan_padded(c.nOut);
  float *run = nullptr;
  SCN_TRY(stream_scratch(s, kScratchChunk, (size_t)std::min(nC - 1, 2) * c.nOutRows * c.Cout * 4 + 16, (void **)&run));
  const float *prev = c.addend;
  for (int i = 0; i < nC; i++) {
    const int k0 = i * kChunkOffsets, Kc = std::min(kChunkOffsets, K - k0);
    const bool last = i == nC - 1;
    TcConv ch = c;
    ch.out = last ? c.out : run + (size_t)(i & 1) * c.nOutRows * c.Cout;
    // W: [K][CinW][Cout] (or [K][Cout][CinW] transposed): CinW x Cout floats per offset.  Offset-reversed operands (wT = 2): offset j
    // of this chunk is W[K - 1 - k0 - j], i.e. the reversal of the block W[K - k0 - Kc, K - k0)
    ch.W = c.W + (size_t)(c.wT == 2 ? K - k0 - Kc : k0) * CinW * c.Cout;
    ch.nbr = c.nbr + (size_t)k0 * nPad;
    ch.tileMask = c.tileMask + (size_t)i * (nPad / 128);
    ch.K = ch.nWeights = Kc;
    ch.bias = i == 0 ? c.bias : nullptr; ch.addend = prev;
    if (!last) { ch.out16 = nullptr; ch.fuse.lat.in = nullptr; ch.fuse.stats = nullptr; } // (the padded input rows go to every chunk)
    ++g_counters[kCntChunkedLaunch];
    SCN_TRY(launch_conv_plan_tc(ch, s));
    prev = ch.out;
  }
  return 0;
}
// A layer of more than 256 output channels (the N of one tcgen05.mma, and half the TMEM columns of an SM) runs as ceil(Cout / 256)
// launches over column slabs of balanced widths, multiples of 32 (320 = 160 + 160, 288 = 160 + 128, 1024 = 4 x 256).  Each slab is
// an ordinary launch of <= 256 columns that writes its columns of the full-width rows (TcParams::ldo), with its own weight image
// (the slab's output columns only), its columns of the bias, of the caller's addend, of the 16-bit copy and of the lateral weight.
// The epilogue BatchNorm statistics (<= kFusedStatsC channels) are not taken.  A chunked plan (K > 64) splits into chunks first,
// and each chunk into slabs.
static int launch_conv_plan_tc_slabs(const TcConv &c, cudaStream_t s) {
  SCN_CHECK(c.Cout % 32 == 0 && c.Cout <= 1024 && c.ldOut == 0, "tcgen05 path: more than 256 output channels need a multiple of 32, at most 1024");
  TcConv b = c;
  b.ldOut = c.Cout;
  b.fuse.stats = nullptr;
  if (half_mode(c.mathMode) && c.Cin % 64 == 0 && !c.in16 && c.nInRows) { // 16-bit operands: one copy of the input rows for all slabs
    void *p = nullptr;
    SCN_TRY(stream_scratch(s, kScratchBf16, (size_t)c.nInRows * c.Cin * 2 + 16, &p));
    SCN_CUDA(launch_to_16(c.in, p, c.nInRows * c.Cin / 4, c.mathMode == kModeF16, s));
    b.in16 = p;
  }
  const int units = c.Cout / 32, n = cdiv(c.Cout, 256);
  for (int i = 0, col = 0; i < n; i++) {
    TcConv sl = b;
    sl.col0 = col;
    sl.Cout = 32 * (units / n + (i < units % n ? 1 : 0));
    SCN_TRY(launch_conv_plan_tc(sl, s));
    col += sl.Cout;
  }
  return 0;
}
// Every conv_plan_tc instantiation the launcher uses: operand type, producer warps, filter offsets per packed atom (G), CTAs per
// SM, deterministic mode.
struct PlanKernel { int op, pw, G, ctas; bool det; void (*fn)(TcParams); };
#define SCN_PLAN(OP, PW, G, CTAS) {OP, PW, G, CTAS, false, conv_plan_tc<OP, PW, G, CTAS, false>}, {OP, PW, G, CTAS, true, conv_plan_tc<OP, PW, G, CTAS, true>}
static const PlanKernel kPlanKernels[] = {
    SCN_PLAN(kOpTF32, 8, 1, 1),   SCN_PLAN(kOpTF32, 4, 1, 2), SCN_PLAN(kOpTF32, 8, 1, 2), SCN_PLAN(kOpTF32X3, 8, 1, 1),
    SCN_PLAN(kOpBF16, 8, 1, 1),   SCN_PLAN(kOpBF16, 4, 1, 2), SCN_PLAN(kOpBF16, 4, 2, 2), SCN_PLAN(kOpBF16, 4, 4, 2),
    SCN_PLAN(kOpBF16, 8, 1, 2),   SCN_PLAN(kOpBF16, 8, 2, 2), SCN_PLAN(kOpBF16, 8, 4, 2),
    SCN_PLAN(kOpF16, 8, 1, 1),    SCN_PLAN(kOpF16, 4, 1, 2),  SCN_PLAN(kOpF16, 4, 2, 2),  SCN_PLAN(kOpF16, 4, 4, 2),
    SCN_PLAN(kOpF16, 8, 1, 2),    SCN_PLAN(kOpF16, 8, 2, 2),  SCN_PLAN(kOpF16, 8, 4, 2)};
#undef SCN_PLAN
int launch_conv_plan_tc(const TcConv &c, cudaStream_t s) {
  const int nOut = c.nOut, K = c.K, Cin = c.Cin, Cout = c.Cout, CinW = c.CinW ? c.CinW : c.Cin;
  if (nOut == 0) return 0;
  if (K > 64 && !c.tileW) {
    SCN_CHECK(c.nbr && c.tileMask && c.nWeights == K && K <= kMaxFilterVolume, "tcgen05 path: wide plan");
    return launch_conv_plan_tc_chunked(c, s);
  }
  const bool f16 = c.mathMode == kModeF16; // 16-bit operands and copies are fp16 (else bf16)
  const bool canPack = half_mode(c.mathMode) && !c.tileW && Cout <= 128 && !c.ldOut; // packed narrow rows: two-CTA configuration only, no column slabs
  if (canPack && CinW == Cin && Cin != 16 && Cin % 32 != 0) {
    // bf16 / fp16 mode, odd channel counts (e.g. the 9-channel network input): 16-bit rows zero-padded to 16 channels (packed, G = 4),
    // 32 channels (G = 2) or a multiple of 64 (whole atoms), written by one pass; the weight image pads itself
    const int Cp = Cin < 16 ? 16 : (Cin < 32 ? 32 : (Cin + 63) / 64 * 64);
    TcConv p = c;
    void *xp = nullptr;
    if (c.fuse.pad16 && c.fuse.padC == Cp) {
      xp = const_cast<void *>(c.fuse.pad16); // the producer already wrote the padded copy
    } else {
      SCN_TRY(stream_scratch(s, kScratchBf16, (size_t)c.nInRows * Cp * 2 + 16, &xp));
      launch_pad_rows16(c.in, xp, c.nInRows, Cin, Cp, f16, s);
    }
    p.in16 = xp; p.Cin = Cp; p.CinW = Cin;
    return launch_conv_plan_tc(p, s);
  }
  if (Cin % 32 != 0 && !(canPack && Cin == 16)) { // rows zero-padded to a multiple of 32 channels (the weight image pads itself)
    const int Cp = (Cin + 31) / 32 * 32;
    float *xp = nullptr;
    SCN_TRY(stream_scratch(s, kScratchPad, (size_t)c.nInRows * Cp * 4 + 16, (void **)&xp));
    k_pad_rows<<<stream_grid(c.nInRows * Cp, 256), 256, 0, LS(s)>>>(c.in, xp, c.nInRows, Cin, Cp);
    TcConv p = c;
    p.in = xp; p.in16 = nullptr; p.Cin = Cp; p.CinW = Cin;
    return launch_conv_plan_tc(p, s);
  }
  if (Cout > 256) return launch_conv_plan_tc_slabs(c, s);
  SCN_CHECK(Cout % 16 == 0 && Cout >= 16 && Cout <= 256 && K <= 64, "tcgen05 path: unsupported channel counts");
  const int ldo = c.ldOut ? c.ldOut : Cout, col0 = c.col0; // (a column slab: columns [col0, col0 + Cout) of rows ldo wide)
  static int envT = -1, envS = -1, envDbg = 0, envProf = 0, envCtas = 0;
  if (envT < 0) {
    envCtas = getenv("SCN_TC_CTAS") ? atoi(getenv("SCN_TC_CTAS")) : 0;
    envT = getenv("SCN_TC_T") ? atoi(getenv("SCN_TC_T")) : 0;
    envS = getenv("SCN_TC_S") ? atoi(getenv("SCN_TC_S")) : 0;
    envDbg = getenv("SCN_TC_DBG") ? atoi(getenv("SCN_TC_DBG")) : 0;
    envProf = getenv("SCN_TC_PROF") ? atoi(getenv("SCN_TC_PROF")) : 0;
  }
  TcParams P;
  P.in = reinterpret_cast<const unsigned char *>(c.in); P.nbr = c.nbr; P.outRow = c.outRow; P.tileMask = c.tileMask; P.tileW = c.tileW;
  P.out = c.out ? c.out + col0 : nullptr; P.bias = c.bias ? c.bias + col0 : nullptr; P.addend = c.addend ? c.addend + col0 : nullptr;
  P.out16 = c.out16 ? static_cast<unsigned char *>(c.out16) + (size_t)col0 * 2 : nullptr;
  P.nOut = nOut; P.K = K; P.Cout = Cout; P.ldo = ldo;
  // bf16 / fp16 mode: rows of >= 64 channels are whole 128-byte atoms; 32- and 16-channel rows (64 / 32 bytes) are PACKED, G = 2 / 4
  // filter offsets side by side in one atom: half / a quarter of the stages, gather bytes and MMAs of the 128-byte-row layout
  const int packG = (canPack && (Cin == 32 || Cin == 16)) ? 64 / Cin : 1;
  P.bf16 = (half_mode(c.mathMode) && (Cin % 64 == 0 || packG > 1)) ? 1 : 0; // 16-bit operands (fp16 in mode 5); other narrow layers keep TF32 operands
  P.f16 = f16 && !P.bf16; // (a TF32-operand launch in fp16 mode writes its 16-bit copy as fp16)
  // TF32X3: the fp32 rows split into two TF32 operands (one-CTA configuration, stages twice as large)
  const int op = P.bf16 ? (f16 ? kOpF16 : kOpBF16) : (c.mathMode == 3 ? kOpTF32X3 : kOpTF32);
  const bool x3 = op == kOpTF32X3;
  void *tmp16 = nullptr;
  if (P.bf16) {
    const void *in16 = c.in16;
    if (!in16) {
      SCN_TRY(stream_scratch(s, kScratchBf16, (size_t)c.nInRows * Cin * 2 + 16, &tmp16));
      if (c.nInRows) SCN_CUDA(launch_to_16(c.in, tmp16, c.nInRows * Cin / 4, f16, s));
      in16 = tmp16;
    }
    P.in = static_cast<const unsigned char *>(in16);
  }
  P.rowBytes = Cin * (P.bf16 ? 2 : 4);
  P.nAtoms = packG > 1 ? 1 : P.rowBytes / 128;
  P.KG = (K + packG - 1) / packG;
  P.nTiles = cdiv(nOut, kTileM);
  P.dbg = envDbg;
  // Tiles per work item: as many as TMEM holds (T x Cout <= 512 columns) so that a weight atom is
  // fetched once per T tiles, but never so many that fewer than ~2 items per SM remain; small levels
  // use 1-tile items and split the filter offsets over CTAs so the whole chip works on them.
  // two CTAs per SM (each with 256 TMEM columns and half the shared memory) unless the layer is too wide for that
  int ctas = envCtas ? envCtas : 2;
  if (Cout > 128) ctas = 1;
  if (packG > 1) ctas = 2;
  // Small levels (at most one tile per SM): nothing else runs beside them, so one CTA per SM with the whole shared memory as
  // a deep ring (up to 6 stages) and 8 producer warps hides the gather latency of the serial offset loop far better than two
  // half-sized CTAs that would mostly stay unused.
  static int smallOne = -1;
  if (smallOne < 0) smallOne = getenv("SCN_TC_SMALL_ONE") ? atoi(getenv("SCN_TC_SMALL_ONE")) : 1;
  if (smallOne && !envCtas && packG == 1 && cdiv(nOut, kTileM) <= kSMs) ctas = 1;
  if (x3) ctas = 1; // (with half the shared memory, a 128-channel layer would not even fit two stages of one tile)
  P.tmemCols = ctas == 2 ? 256 : 512;
  const size_t smemBudget = ctas == 2 ? ((233472 - kBuildRoom) / 2 - 1024) : (227 * 1024 - kBuildRoom);
  const int Tcap = std::min(packG == 4 ? 2 : kMaxT, P.tmemCols / Cout);
  const size_t fixed = kEpiBytes + 64 * 8 + 64;
  const size_t stageMul = x3 ? 2 : 1; // TF32X3: hi and lo atoms of A and of W
  auto ring = [&](int t) { return (int)((smemBudget - fixed) / (stageMul * ((size_t)t * kAtomBytes + (size_t)Cout * 128))); };
  int T = Tcap;
  if (ctas == 1) while (T > 2 && ring(T) < 3) T--; // a 2-slot ring exposes the gather latency (measured: T=3/S=3 beats T=4/S=2 by 12 %)
  while (T > 1 && ring(T) < 2) T--;
  while (T > 1 && cdiv(P.nTiles, T) < 2 * kSMs * ctas) T--;
  if (c.tileW) T = 1;
  if (envT > 0 && envT <= Tcap && !c.tileW && ring(envT) >= 2) T = envT; // (a forced T must leave room for a 2-stage ring)
  P.T = T;
  P.nAcc = 2 * T * Cout <= P.tmemCols ? 2 : 1;
  P.nSuper = cdiv(P.nTiles, P.T);
  P.kSplit = 1;
  // Only really small levels (<= kSplitMaxItems items) spread the filter offsets of an item over CTAs: the split costs a memset,
  // atomic accumulation and a separate bf16 pass, and rules out the BatchNorm statistics in the epilogue; from a few dozen
  // items on, one CTA per item doing all offsets is as fast and needs one launch instead of three.
  static int kSplitMaxItems = -1;
  if (kSplitMaxItems < 0) kSplitMaxItems = getenv("SCN_TC_SPLIT_MAX") ? atoi(getenv("SCN_TC_SPLIT_MAX")) : 40;
  if (P.nSuper <= kSplitMaxItems && !c.tileW) P.kSplit = std::max(1, std::min(packG > 1 ? P.KG : K, kSMs * ctas / P.nSuper));
  P.stats = nullptr;
  P.statsPart = nullptr;
  P.part = nullptr;
  const bool det = deterministic();
  if (c.fuse.stats && P.kSplit == 1 && Cout <= kFusedStatsC && Cout % 32 == 0) { P.stats = c.fuse.stats; if (c.fused) c.fused->stats = true; ++g_counters[kCntEpilogueStats]; }
  if (P.stats) { // deterministic mode: per-(item, epilogue warp) sums, added in item order after the launch
    if (det) SCN_TRY(det_scratch(s, (size_t)P.nSuper * 4 * 2 * Cout * sizeof(double), (void **)&P.statsPart));
    else ++g_counters[kCntFloatAtomic];
  }
  const size_t stageBytes = stageMul * ((size_t)P.T * kAtomBytes + (size_t)Cout * 128);
  P.S = (int)std::min<size_t>(envS > 0 ? envS : 6, (smemBudget - fixed) / stageBytes);
  SCN_CHECK(P.S >= 2, "tcgen05 path: shared memory budget exceeded");
  static int envLag = -2;
  if (envLag == -2) envLag = getenv("SCN_TC_LAG") ? atoi(getenv("SCN_TC_LAG")) : -1;
  P.lag = std::max(0, std::min(3, envLag >= 0 ? envLag : P.S - 2));
  if (P.lag > P.S - 2) P.lag = std::max(0, P.S - 2);
  const size_t smem = (size_t)P.S * stageBytes + fixed;
  SCN_CHECK(c.out || (P.kSplit == 1 && c.out16), "tcgen05 path: fp32 output dropped on a launch that needs it");
  ++g_counters[kCntTcLaunch];
  if (x3) ++g_counters[kCntTf32x3Launch];
  if (op == kOpF16) ++g_counters[kCntF16Launch];
  if (P.kSplit > 1) ++g_counters[kCntSplitLaunch];
  if (P.kSplit > 1 && det) SCN_TRY(det_scratch(s, (size_t)P.kSplit * nOut * Cout * 4, (void **)&P.part)); // (k_split_sum writes every output row)
  else if (P.kSplit > 1 && ldo == Cout) { ++g_counters[kCntFloatAtomic]; SCN_CUDA(cudaMemsetAsync(c.out, 0, (size_t)nOut * Cout * 4, s)); }
  else if (P.kSplit > 1) { ++g_counters[kCntFloatAtomic]; SCN_CUDA(cudaMemset2DAsync(P.out, (size_t)ldo * 4, 0, (size_t)Cout * 4, nOut, s)); } // (the slab's columns only)
  unsigned char *wimg = nullptr;
  bool wimgOwned = false;
  const int el16 = f16 ? kWimgF16 : kWimgBF16; // element format of a 16-bit image
  SCN_TRY(get_wimg(c.W, c.wTag, c.nWeights, Cin, CinW, Cout, packG > 1 ? el16 + 16 * packG : x3 ? kWimgSplit : P.bf16 ? el16 : 0, s, &wimg, &wimgOwned, c.wT, col0, ldo));
  P.wimg = wimg;
  P.in2 = nullptr; P.wimg2 = nullptr; P.rowBytes2 = 0; P.nAtoms2 = 0;
  unsigned char *wimg2 = nullptr;
  bool wimg2Owned = false;
  const Lateral &lat = c.fuse.lat; // taken when the launch is a whole-atom (unpacked) tensor-core launch
  if (lat.in && packG == 1 && K < kLateralBit && lat.rows > 0 && (!P.bf16 || lat.in16)) {
    const int esz = P.bf16 ? 2 : 4, per = 128 / esz, C2 = lat.Cin; // per = channels of one K atom
    if ((C2 * esz) % 16 == 0) {
      const int C2p = (C2 + per - 1) / per * per;
      SCN_TRY(get_wimg(lat.w, lat.tag, 1, C2p, C2, Cout, x3 ? kWimgSplit : P.bf16 ? el16 : 0, s, &wimg2, &wimg2Owned, 0, col0, ldo));
      P.in2 = static_cast<const unsigned char *>(P.bf16 ? lat.in16 : static_cast<const void *>(lat.in));
      P.rowBytes2 = C2 * esz;
      P.nAtoms2 = C2p / per;
      P.wimg2 = wimg2;
      if (c.fused) c.fused->lateral = true;
      ++g_counters[kCntLateralFolded];
    }
  }
  static bool attr = false;
  if (!attr) {
    const int half = (233472 - kBuildRoom) / 2 - 1024;
    for (const PlanKernel &k : kPlanKernels) SCN_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, k.ctas == 1 ? 227 * 1024 : half));
    attr = true;
  }
  static int envSms = -1;
  if (envSms < 0) envSms = getenv("SCN_TC_SMS") ? atoi(getenv("SCN_TC_SMS")) : kSMs;
  const int grid = std::min(P.nSuper * P.kSplit, std::min(kSMs, envSms) * ctas);
  static int envDyn = -1;
  if (envDyn < 0) envDyn = getenv("SCN_TC_DYNAMIC") ? atoi(getenv("SCN_TC_DYNAMIC")) : 0; // measured on B470: dominant layer 0.536 (dynamic) vs 0.545 ms (static), whole forward 5.0-5.1 vs 4.92 ms -> static stride stays the default
  P.sched = nullptr;
  if (envDyn && P.nSuper * P.kSplit > grid) SCN_TRY(sched_counters(s, &P.sched)); // (one item per CTA: nothing to balance)
  P.prof = nullptr;
  if (envProf) {
    SCN_CUDA(cudaMallocAsync((void **)&P.prof, 2 * kSMs * 32 * 8, s));
    SCN_CUDA(cudaMemsetAsync(P.prof, 0, 2 * kSMs * 32 * 8, s));
  }
  // producer warps of the two-CTA configuration: 4 (96 registers) or 8 (72 registers); bit 0 = packed layers, bit 1 = whole-atom layers
  static int envPw8 = -1;
  if (envPw8 < 0) envPw8 = getenv("SCN_TC_PW8") ? atoi(getenv("SCN_TC_PW8")) : 0;
  const int pw = ctas == 1 || (packG > 1 && (envPw8 & 1)) || (packG == 1 && (envPw8 & 2)) ? 8 : 4;
  const PlanKernel *kern = nullptr;
  for (const PlanKernel &k : kPlanKernels)
    if (k.op == op && k.pw == pw && k.G == packG && k.ctas == ctas && k.det == det) kern = &k;
  SCN_CHECK(kern, "tcgen05 path: no kernel instantiated for this configuration");
  // warps: 4 epilogue, the producers, the MMA issuer, the weight loader (and the TF32X3 splitters)
  SCN_CUDA(launch_pdl(kern->fn, dim3(grid), dim3(32 * (4 + pw + 2 + (x3 ? kSplitWarps : 0))), smem, LS(s), P));
  SCN_CUDA(cudaGetLastError());
  if (envProf) { // developer aid: mean stall cycles per role over the CTAs of this launch
    static long long h[2 * kSMs * 32];
    SCN_CUDA(cudaMemcpyAsync(h, P.prof, sizeof h, cudaMemcpyDeviceToHost, s));
    SCN_CUDA(cudaStreamSynchronize(s));
    double m[32] = {0};
    for (int b = 0; b < grid; b++) for (int i = 0; i < 32; i++) m[i] += (double)h[b * 32 + i] / grid;
    fprintf(stderr, "[tcprof] ctas=%d pw=%d grid=%d T=%d K=%d Cin=%d Cout=%d S=%d lag=%d nAcc=%d kSplit=%d | epi total %.0f waitAcc %.0f | prod total %.0f empty %.0f cpwait %.0f stages %.0f | mma total %.0f accEmpty %.0f full %.0f stages %.0f issue %.0f commit %.0f | bld total %.0f empty %.0f\n",
            ctas, pw, grid, P.T, K, Cin, Cout, P.S, P.lag, P.nAcc, P.kSplit, m[0], m[1], m[4], m[5], m[6], m[7], m[10], m[11], m[12], m[13], m[14], m[15], m[16], m[17]);
    cudaFreeAsync(P.prof, s);
  }
  if (P.statsPart) SCN_TRY(ordered_sum(P.statsPart, P.nSuper * 4, 2l * Cout, P.stats, s, Cout, kFusedStatsC)); // into replica 0
  if (P.part) // the split partials in split order, and the 16-bit copy from the same registers
    SCN_CUDA(launch_pdl(f16 ? k_split_sum<true> : k_split_sum<false>, dim3(stream_grid((long)nOut * Cout / 4, 256)), dim3(256), 0, LS(s),
                        reinterpret_cast<const float4 *>(P.part), P.kSplit, (long)nOut * Cout / 4, Cout / 4, Cout / 4, ldo / 4, reinterpret_cast<float4 *>(P.out),
                        static_cast<uint2 *>(P.out16)));
  else if (c.out16 && P.kSplit > 1 && c.nOutRows > 0 && ldo == Cout) // partial sums were accumulated atomically: the 16-bit copy needs the finished rows
    SCN_CUDA(launch_to_16(c.out, c.out16, c.nOutRows * Cout / 4, f16, s));
  else if (c.out16 && P.kSplit > 1 && c.nOutRows > 0) // (the same for the columns of a slab)
    SCN_CUDA(launch_pdl(f16 ? k_split_sum<true> : k_split_sum<false>, dim3(stream_grid(c.nOutRows * Cout / 4, 256)), dim3(256), 0, LS(s),
                        reinterpret_cast<const float4 *>(P.out), 1, c.nOutRows * Cout / 4, Cout / 4, ldo / 4, ldo / 4, static_cast<float4 *>(nullptr),
                        static_cast<uint2 *>(P.out16)));
  if (wimgOwned) cudaFreeAsync(wimg, s);
  if (wimg2Owned) cudaFreeAsync(wimg2, s);

  return 0;
}

// ====================================================================== weight gradient on the tensor cores
//   dW[k] = sum over the rules (i, o) of filter offset k of   in[i]^T (Cin x 1)  *  dOut[o] (1 x Cout)
// = a GEMM with M = Cin, N = Cout and the RULES as the reduction dimension.  The gathered rows land in shared memory
// exactly as in the forward kernel (one 128-byte swizzled row per rule and 64-channel block); read as an MN-MAJOR
// operand (instruction descriptor bits 15 / 16, shared-memory descriptor LBO = distance between channel blocks, SBO =
// 1024 B between groups of 8 rules) the very same bytes are the transposed matrices the product needs -- no transpose
// pass, both operands are plain row gathers.  Replaces dConvolution_KMxKN_backward_dW_A/B (SCN/CUDA/Convolution.cu:249-410).
// Producer side of both weight-gradient kernels: one warp requests its RW rows of a stage (4 rows per instruction, 8 lanes x 16 B per
// 128-byte block of a row).  Straight-line code: the kernels are paced by how fast 8 producer warps can issue these requests
// (measured with run-time block loops: ~1000 instructions per warp and stage, 3 us per stage, every memory pipe below 10 %).
// maskA / maskB: bit b = this lane's 16-byte chunk of block b exists in a row (narrow rows end inside a block); blocks that lie
// entirely beyond the row (the zero padding of M to 128) are zeroed once at kernel start and never written again.
struct DwLane { uint32_t maskA, maskB, chunkOff; int nBaReal, nBb; };
__device__ __forceinline__ DwLane dw_lane(int rowBytesA, int rowBytesB, int lane) {
  DwLane L;
  L.chunkOff = (uint32_t)(lane & 7) * 16u;
  L.nBaReal = (rowBytesA + 127) / 128;
  L.nBb = (rowBytesB + 127) / 128;
  L.maskA = 0; L.maskB = 0;
#pragma unroll
  for (int b = 0; b < 4; b++) {
    if (b * 128 + (int)L.chunkOff < rowBytesA) L.maskA |= 1u << b;
    if (b * 128 + (int)L.chunkOff < rowBytesB) L.maskB |= 1u << b;
  }
  return L;
}
// one operand of a stage: the RW rows of this warp, ids in lanes 0..RW-1 (replicated every RW lanes); rows of rowBytes, ld bytes apart
// (ld > rowBytes: a channel block of wider rows)
template <int RW>
__device__ __forceinline__ void dw_fill_operand(const unsigned char *base, int rowBytes, int ld, int nB, uint32_t mask, uint32_t chunkOff, int ids, uint32_t sOp,
                                                uint32_t blockBytes, int pw, int lane) {
  if (rowBytes <= 64) {
    // Narrow rows (64 / 32 bytes = 32 / 16 bf16 channels): 4 / 2 lanes per row, 8 / 16 rows per instruction instead of 4 -- only the
    // chunks that exist are written, the rest of the 128-byte row stays zero from the start of the launch (dw_zero_padding).
    const int cpr = rowBytes >> 4, sh = cpr == 4 ? 2 : 1; // chunks per row (power of two), log2
    const int ch = lane & (cpr - 1), rs = lane >> sh, rpi = 32 >> sh;
#pragma unroll 1
    for (int i = 0; i < RW; i += rpi) {
      const int rl = i + rs;
      const bool mine = rl < RW;
      const int id = __shfl_sync(0xffffffffu, ids, mine ? rl : 0);
      const int row = pw * RW + rl;
      if (mine) cp_async16(sOp + (uint32_t)row * 128u + ((uint32_t)(ch ^ (row & 7)) << 4), base + (size_t)max(id, 0) * ld + ch * 16, id >= 0 ? 16u : 0u);
    }
    return;
  }
  const int chunk = lane & 7, rsub = lane >> 3;
#pragma unroll 2
  for (int i = 0; i < RW / 4; i++) {
    const int rl = i * 4 + rsub;
    const int id = __shfl_sync(0xffffffffu, ids, rl);
    const int row = pw * RW + rl;
    const uint32_t dst = sOp + (uint32_t)row * 128u + ((uint32_t)(chunk ^ (row & 7)) << 4);
    const unsigned char *pr = base + (size_t)max(id, 0) * ld;
    const uint32_t ok = id >= 0 ? 16u : 0u;
#pragma unroll 1
    for (int b = 0; b < nB; b++) {
      const bool v = (mask >> b) & 1u; // this lane's chunk of block b lies inside the row
      cp_async16(dst + (uint32_t)b * blockBytes, pr + (v ? (uint32_t)b * 128u + chunkOff : 0u), v ? ok : 0u);
    }
  }
}
template <int RW>
__device__ __forceinline__ void dw_fill_stage(const DwLane &L, const unsigned char *A, const unsigned char *B, int rowBytesA, int rowBytesB, int ldA, int ldB, int srcId,
                                              int dstId, uint32_t sbase, uint32_t blockBytes, int nBa, int pw, int lane) {
  static_assert(RW >= 4 && RW % 4 == 0, "a producer warp requests 4 rows per instruction");
  // Rolled loops with everything loop-invariant hoisted: ~10 instructions per copy.  (Fully unrolled with per-copy predicates the
  // compiler produced ~40 instructions per copy, ~800 per warp and stage, and the producer warps' issue rate set the pace.)
  dw_fill_operand<RW>(A, rowBytesA, ldA, L.nBaReal, L.maskA, L.chunkOff, srcId, sbase, blockBytes, pw, lane);
  dw_fill_operand<RW>(B, rowBytesB, ldB, L.nBb, L.maskB, L.chunkOff, dstId, sbase + (uint32_t)nBa * blockBytes, blockBytes, pw, lane);
}
// Zero the whole stage ring once per launch: the blocks that hold the channel padding of A (rows narrower than 256 bytes) and the
// chunks of a 128-byte row beyond a narrow row's end are never written by the producers and read (as zeros) by every MMA.
__device__ __forceinline__ void dw_zero_padding(unsigned char *sStage, int S, uint32_t stageBytes, uint32_t blockBytes, int nBaReal, int nBa) {
  uint4 *q = reinterpret_cast<uint4 *>(sStage);
  const uint32_t n = (uint32_t)S * stageBytes / 16u;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) q[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async(); // generic-proxy writes -> the tensor core's (async proxy) reads
}
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t addr, uint32_t lboBytes);
// MMA issue of one weight-gradient stage: NJ x nMh instructions as straight-line code from precomputed descriptors.  The issuing
// warp, not the memory system, paced these kernels: with run-time loop bounds and an integer division per instruction it spent
// ~3000 cycles per stage on 8 instructions (SCN_DW_PROF: wait-full 7 % of the MMA warp's time, producers waiting 15 %).
template <bool BF16, int NJ>
__device__ __forceinline__ void dw_issue_stage(uint32_t sbase, uint32_t blockBytes, int nBa, int nMh, uint32_t aBlkStride16, uint32_t tmemD, int Cout, uint32_t idesc, bool first) {
  constexpr uint32_t kStep16 = (uint32_t)(BF16 ? 16 : 8) * 128u >> 4; // descriptor address units (16 B) per instruction along the rule dimension
  const uint64_t a0 = smem_desc_mn_sw128(sbase, blockBytes), b0 = smem_desc_mn_sw128(sbase + (uint32_t)nBa * blockBytes, blockBytes);
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    tc_mma<BF16>(tmemD, a0 + (uint64_t)(j * kStep16), b0 + (uint64_t)(j * kStep16), idesc, (!first || j > 0) ? 1u : 0u);
    if (nMh > 1) tc_mma<BF16>(tmemD + (uint32_t)Cout, a0 + (uint64_t)(aBlkStride16 + j * kStep16), b0 + (uint64_t)(j * kStep16), idesc, (!first || j > 0) ? 1u : 0u);
  }
}
constexpr int kDwProd = 16; // producer warps of the weight-gradient kernels (their request issue rate paces the kernels: 8 -> 16 measured below)
// One CTA per SM: 4 epilogue warps (TMEM -> red.global.add), 8 producer warps, 1 MMA warp; a work item is a chunk of
// one offset's rule list, its partial dW[k] is accumulated in TMEM and added to global memory once.
struct DwParams {
  const unsigned char *a, *b; // operand-typed rows: `in` (rowBytesA per row, ldA apart) and `d_out` (rowBytesB, ldB apart)
  const int2 *pairs;
  const int *d_off;           // K + 1 list offsets
  float *dW;
  float *part;                // deterministic mode: [item][Cin][Cout], item w's partial dW[w % K] (plain stores), summed in part order afterwards
  int K, Cin, Cout, nC, srcIsY, rowBytesA, rowBytesB, R, S, nAcc; // nC: parts per rule list
  // a channel block of a wider layer (launch_conv_dw_tc): rows ldA / ldB bytes apart, and dW / part rows ldW floats apart, offsets
  // (and work-item slots) wStride floats apart; Cin x Cout, rowBytes and wStride = Cin Cout otherwise
  int ldA, ldB, ldW;
  long wStride;
};
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t addr, uint32_t lboBytes) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lboBytes >> 4) & 0x3fffu) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// BF16: 16-bit operands (kind::f16), fp16 ones with F16 (math mode 5), else TF32
template <bool BF16, bool F16 = false>
__global__ void __launch_bounds__(32 * (5 + kDwProd), 1) conv_dw_tc(const DwParams P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // `in` rows narrower than 128 channels are zero-padded to M = 128 in shared memory (zero-filled chunks, no traffic)
  const int R = P.R, nBa = max(P.rowBytesA, 256) / 128, nBb = (P.rowBytesB + 127) / 128;
  const uint32_t blockBytes = (uint32_t)R * 128u, stageBytes = (uint32_t)(nBa + nBb) * blockBytes;
  unsigned char *sStage = smem;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sStage + (size_t)P.S * stageBytes);
  uint64_t *full = bars, *empty = bars + P.S, *accFull = bars + 2 * P.S, *accEmpty = accFull + 2;
  uint32_t *tmemSlot = reinterpret_cast<uint32_t *>(accEmpty + 2);
  if (tid == 0) {
    for (int i = 0; i < P.S; i++) { mbar_init(smem_u32(full + i), kDwProd * 32); mbar_init(smem_u32(empty + i), 1); }
    for (int i = 0; i < 2; i++) { mbar_init(smem_u32(accFull + i), 1); mbar_init(smem_u32(accEmpty + i), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  dw_zero_padding(sStage, P.S, stageBytes, blockBytes, (P.rowBytesA + 127) / 128, nBa);
  constexpr int kMmaWarp = 4 + kDwProd;
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmemSlot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmemBase = *tmemSlot;
  const int nItems = P.K * P.nC;
  const int nMh = (P.Cin + 127) / 128, accCols = nMh * P.Cout;
  // item w -> (list k = w % K, part c = w / K of nC): the rules [len c / nC, len (c + 1) / nC) of list k.  The lists are in row
  // order, so part c of every list covers about the same region of the grid, and the ~148 items in flight at any time are
  // all 27 offsets of a few neighbouring parts: their rows stay in L2 across the offsets.  (List-major order swept the whole grid
  // once per offset: 4.3 GB of DRAM reads for 5.6 GB of requests on the 128 -> 128 level-0 layer, 81 % of the HBM peak.)
  auto item = [&](int w, int &k, int &r0, int &cnt) {
    const int c = w / P.K;
    k = w - c * P.K;
    const int lo = __ldg(P.d_off + k), hi = __ldg(P.d_off + k + 1);
    const long len = hi - lo;
    r0 = lo + (int)(len * c / P.nC);
    cnt = lo + (int)(len * (c + 1) / P.nC) - r0; // may be 0 (a short list): every role skips such an item
  };
  if (warp < 4) {
    // ---------------- epilogue: partial dW[k] of the item -> global memory (fp32 reductions)
    int itN = 0;
    for (int w = blockIdx.x; w < nItems; w += gridDim.x) {
      int k, r0, cnt;
      item(w, k, r0, cnt);
      if (cnt <= 0) {
        if (P.part) // (an empty part still owns a slot of the ordered sum)
          for (long i = tid; i < (long)P.Cin * P.Cout; i += 128) P.part[(size_t)w * P.wStride + i / P.Cout * P.ldW + i % P.Cout] = 0.f;
        continue;
      }
      const int it = itN++;
      const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
      mbar_wait(smem_u32(accFull + a), use & 1);
      tc_fence_after();
      for (int mh = 0; mh < nMh; mh++) {
        const int ci = mh * 128 + warp * 32 + lane;
        float *dst = (P.part ? P.part + (size_t)w * P.wStride : P.dW + (size_t)k * P.wStride) + (size_t)ci * P.ldW;
        if (mh * 128 + warp * 32 >= P.Cin) continue; // rows of the channel padding (warp-uniform)
        for (int c0 = 0; c0 < P.Cout; c0 += 32) {
          uint32_t v[32];
          tmem_ld(tmemBase + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * accCols + mh * P.Cout + c0), v);
          if (ci < P.Cin && P.part) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4 *>(dst + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          } else if (ci < P.Cin) {
#pragma unroll
            for (int j = 0; j < 32; j++) atomicAdd(dst + c0 + j, __uint_as_float(v[j]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(accEmpty + a));
    }
  } else if (warp < 4 + kDwProd) {
    // ---------------- producers: rows of `in` by the rules' source ids, rows of `d_out` by their destination ids
    const int pw = warp - 4, RW = R / kDwProd; // rules per warp and stage
    const DwLane DL = dw_lane(P.rowBytesA, P.rowBytesB, lane);
    uint32_t slot = 0, round = 0;
    for (int w = blockIdx.x; w < nItems; w += gridDim.x) {
      int k, r0, cnt;
      item(w, k, r0, cnt);
      if (cnt <= 0) continue;
      // the rule ids of a stage are fetched two stages ahead: the dependent chain (ids -> row addresses -> copies) otherwise
      // costs one memory round trip per stage and sets the pace of the whole kernel on narrow layers
      auto load_pair = [&](int base) {
        const int rr = base + pw * RW + (lane & (RW - 1));
        return (base < cnt && rr < cnt) ? __ldg(P.pairs + r0 + rr) : make_int2(-1, -1);
      };
      int2 pr1 = load_pair(0), pr2 = load_pair(R);
      for (int base = 0; base < cnt; base += R) {
        const int2 pr = pr1;
        pr1 = pr2;
        pr2 = load_pair(base + 2 * R);
        const int srcId = P.srcIsY ? pr.y : pr.x, dstId = P.srcIsY ? pr.x : pr.y;
        mbar_wait(smem_u32(empty + slot), (round & 1u) ^ 1u);
        const uint32_t sbase = smem_u32(sStage) + slot * stageBytes;
        if (R == 128) dw_fill_stage<128 / kDwProd>(DL, P.a, P.b, P.rowBytesA, P.rowBytesB, P.ldA, P.ldB, srcId, dstId, sbase, blockBytes, nBa, pw, lane);
        else dw_fill_stage<64 / kDwProd>(DL, P.a, P.b, P.rowBytesA, P.rowBytesB, P.ldA, P.ldB, srcId, dstId, sbase, blockBytes, nBa, pw, lane);
        cp_async_mbar_arrive_noinc(smem_u32(full + slot));
        if (++slot == (uint32_t)P.S) { slot = 0; round++; }
      }
    }
  } else {
    // ---------------- MMA issuer: both operands MN-major (bits 15, 16), M = 128, N = Cout, 32 bytes of K (= 16 bf16 / fp16, 8 tf32 rules) per
    // instruction (kind::f16 takes MN-major operands in fp16 as in bf16)
    const uint32_t fmt = F16 ? 0u : BF16 ? 1u : 2u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(P.Cout >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr int kRulesPerMma = BF16 ? 16 : 8;
    const uint32_t aBlkStride16 = ((uint32_t)(nBa / nMh) * blockBytes) >> 4; // second half of M (channels 128..255): descriptor units
    uint32_t slot = 0, round = 0;
    int itN = 0;
    for (int w = blockIdx.x; w < nItems; w += gridDim.x) {
      int k, r0, cnt;
      item(w, k, r0, cnt);
      if (cnt <= 0) continue;
      const int it = itN++;
      const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
      mbar_wait(smem_u32(accEmpty + a), (use & 1) ^ 1);
      tc_fence_after();
      for (int base = 0; base < cnt; base += R) {
        mbar_wait(smem_u32(full + slot), round & 1u);
        tc_fence_after();
        const uint32_t sbase = smem_u32(sStage) + slot * stageBytes;
        if (elect_one()) {
          if (R == 128) dw_issue_stage<BF16, 128 / kRulesPerMma>(sbase, blockBytes, nBa, nMh, aBlkStride16, tmemBase + (uint32_t)(a * accCols), P.Cout, idesc, base == 0);
          else dw_issue_stage<BF16, 64 / kRulesPerMma>(sbase, blockBytes, nBa, nMh, aBlkStride16, tmemBase + (uint32_t)(a * accCols), P.Cout, idesc, base == 0);
          tc_commit(smem_u32(empty + slot));
        }
        __syncwarp();
        if (++slot == (uint32_t)P.S) { slot = 0; round++; }
      }
      if (elect_one()) tc_commit(smem_u32(accFull + a));
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"(512u) : "memory");
  }
}
// The live tiles of a work item (tiles t0, t0 + step, ... whose mask has bit k), found 32 candidates at a time: every lane reads one
// candidate's mask word, a ballot turns the words into a bit set, and the words of the NEXT 32 candidates are already on their way
// while the current ones are consumed (probing tile by tile cost one dependent memory round trip per candidate).  Whole-warp calls.
struct LiveTiles {
  const unsigned long long *mask;
  int k, t0, t1, step, lane, base;
  unsigned bits;
  unsigned long long ahead; // this lane's mask word of candidate base + 32 + lane
  __device__ __forceinline__ unsigned long long word(int b) const {
    const long t = t0 + (long)(b + lane) * step;
    return t < t1 ? __ldg(mask + t) : 0ull;
  }
  __device__ __forceinline__ void init(const unsigned long long *m, int k_, int t0_, int t1_, int step_, int lane_) {
    mask = m; k = k_; t0 = t0_; t1 = t1_; step = step_; lane = lane_; base = 0;
    const unsigned long long w0 = word(0);
    ahead = word(32);
    bits = __ballot_sync(0xffffffffu, (w0 >> k) & 1ull);
  }
  __device__ __forceinline__ int next() { // the next live tile, or t1 when there is none left
    for (;;) {
      if (bits) { const int j = __ffs(bits) - 1; bits &= bits - 1; return t0 + (base + j) * step; }
      if (t0 + (long)(base + 32) * step >= t1) return t1;
      base += 32;
      bits = __ballot_sync(0xffffffffu, (ahead >> k) & 1ull);
      ahead = word(base + 32);
    }
  }
};
// The same product driven by the OUTPUT-STATIONARY PLAN instead of the per-offset rule lists.  The rule lists are in the
// reference's hash-iteration order, i.e. random in memory: every rule cost two random 64..512-byte DRAM accesses (measured: 1.1 ms
// for each of the three level-0 layers of B470 whatever their width).  The plan lists the same rules tile by tile in spatial block
// order -- (nbr[p][k], outRow[p]) for every plan position p with a neighbour at offset k -- so consecutive rules touch
// neighbouring rows and the gathers hit L2 like the forward pass's.  A work item is (offset k, a range of tiles); a stage is R
// positions of one tile whose mask has bit k set; positions without a neighbour are zero-filled rows (no traffic, no contribution).
struct DwPlanParams {
  const unsigned char *a, *b; // operand-typed rows: `in` (rowBytesA per row) and `d_out` (rowBytesB)
  const int *nbr, *outRow;
  const unsigned long long *tileMask;
  float *dW;
  int K, Cin, Cout, swap, rowBytesA, rowBytesB, R, S, nAcc;
  int nPos, nTiles, chunkTiles, itemsPerK; // plan positions, tiles of 128, tiles per work item, work items per offset
  unsigned *sched; // [0] next work item, [1] CTAs that have drawn their last item (self-resetting, see sched_counters)
  long long *prof; // developer (SCN_DW_PROF): per CTA [0] total, [1] producer wait-empty, [2] producer stages, [3] mma total, [4] mma wait-full, [5] mma wait-acc, [6] epilogue busy
};
template <bool BF16, bool F16 = false>
__global__ void __launch_bounds__(32 * (6 + kDwProd), 1) conv_dw_plan_tc(const DwPlanParams P) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int R = P.R, nBa = max(P.rowBytesA, 256) / 128, nBb = (P.rowBytesB + 127) / 128, nHalf = 128 / R;
  const uint32_t blockBytes = (uint32_t)R * 128u, stageBytes = (uint32_t)(nBa + nBb) * blockBytes;
  unsigned char *sStage = smem;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sStage + (size_t)P.S * stageBytes);
  uint64_t *full = bars, *empty = bars + P.S, *accFull = bars + 2 * P.S, *accEmpty = accFull + 2;
  uint32_t *tmemSlot = reinterpret_cast<uint32_t *>(accEmpty + 2);
  // work items are drawn from a global counter by warp 13 and published to the other 13 warps through a ring in shared memory
  // (the cost of an item -- the live tiles of its offset -- is only known on the device: a static stride left the average CTA idle
  // for 45 % of the launch)
  Sched SC{bars + 24, bars + 24 + kSchedSlots, reinterpret_cast<volatile int *>(bars + 24 + 2 * kSchedSlots)};
  if (tid == 0) {
    for (int i = 0; i < P.S; i++) { mbar_init(smem_u32(full + i), kDwProd * 32); mbar_init(smem_u32(empty + i), 1); }
    for (int i = 0; i < 2; i++) { mbar_init(smem_u32(accFull + i), 1); mbar_init(smem_u32(accEmpty + i), 4); }
    for (int i = 0; i < kSchedSlots; i++) { mbar_init(smem_u32(SC.full + i), 1); mbar_init(smem_u32(SC.empty + i), 5 + kDwProd); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  dw_zero_padding(sStage, P.S, stageBytes, blockBytes, (P.rowBytesA + 127) / 128, nBa);
  constexpr int kMmaWarp = 4 + kDwProd;
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmemSlot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmemBase = *tmemSlot;
  const int nItems = P.K * P.itemsPerK;
  const int nMh = (P.Cin + 127) / 128, accCols = nMh * P.Cout;
  // item -> (offset k, tile range); every role walks the live tiles of the range in the same order
  // Work item w = (offset k = w % K, tile class c = w / K): the tiles c, c + itemsPerK, c + 2 itemsPerK, ...  Every item of an offset
  // samples the whole grid (equal cost within an offset: a contiguous range of a sparse offset may hold no live tile at all) and
  // consecutive items -- the ones a CTA draws with its static stride -- belong to different offsets.
  const int tStep = P.itemsPerK;
  auto item = [&](int w, int &k, int &t0, int &t1) {
    k = w % P.K;
    t0 = w / P.K;
    t1 = P.nTiles;
  };

  if (warp < 4) {
    // ---------------- epilogue: partial dW[k] of the item -> global memory (fp32 reductions)
    int it = 0;
    for (;; it++) {
      const int w = sched_take(SC, it, lane == 0);
      if (w < 0) break;
      int k, t0, t1;
      item(w, k, t0, t1);
      LiveTiles LT;
      LT.init(P.tileMask, k, t0, t1, tStep, lane);
      const bool any = LT.next() < t1;
      const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
      mbar_wait(smem_u32(accFull + a), use & 1);
      tc_fence_after();
      for (int mh = 0; any && mh < nMh; mh++) {
        const int ci = mh * 128 + warp * 32 + lane;
        float *dst = P.dW + ((size_t)k * P.Cin + ci) * P.Cout;
        if (mh * 128 + warp * 32 >= P.Cin) continue; // rows of the channel padding (warp-uniform)
        for (int c0 = 0; c0 < P.Cout; c0 += 32) {
          uint32_t v[32];
          tmem_ld(tmemBase + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * accCols + mh * P.Cout + c0), v);
          if (ci < P.Cin) {
#pragma unroll
            for (int j = 0; j < 32; j++) atomicAdd(dst + c0 + j, __uint_as_float(v[j]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(accEmpty + a));
    }
  } else if (warp < 4 + kDwProd) {
    // ---------------- producers: rows of `in` by the plan's neighbour ids, rows of `d_out` by its output rows (swapped for a deconvolution)
    const int pw = warp - 4, RW = R / kDwProd; // positions per warp and stage
    const DwLane DL = dw_lane(P.rowBytesA, P.rowBytesB, lane);
    uint32_t slot = 0, round = 0;
    long long pwait = 0, pstages = 0;
    const long long pt0 = P.prof ? clock64() : 0;
    for (int itp = 0;; itp++) {
      const int w = sched_take(SC, itp, lane == 0);
      if (w < 0) break;
      int k, t0, t1;
      item(w, k, t0, t1);
      // (both loads are independent of each other's result: the ids of the next two stages are in flight while this stage's rows are requested)
      auto load_ids = [&](int t, int h, int &idn, int &ido) { // lane l holds position h R + pw RW + l % RW of tile t
        idn = -1; ido = -1;
        if (t >= t1) return;
        const int r = h * R + pw * RW + (lane & (RW - 1));
        const long p = (long)t * 128 + r;
        idn = __ldg(P.nbr + ((size_t)t * P.K + k) * 128 + r);
        ido = p < P.nPos ? (P.outRow ? __ldg(P.outRow + p) : (int)p) : -1;
      };
      LiveTiles LT;
      LT.init(P.tileMask, k, t0, t1, tStep, lane);
      // three stages in flight: (t, h) is being filled, (tB, hB) and (tA, hA) are the next two, their ids already requested
      auto advance = [&](int &t, int &h) { if (++h == nHalf) { h = 0; t = LT.next(); } };
      int t = LT.next(), h = 0;
      int tB = t, hB = h, tA, hA, idn1, ido1, idn2, ido2;
      load_ids(t, h, idn1, ido1);
      if (tB < t1) advance(tB, hB);
      tA = tB; hA = hB;
      load_ids(tB, hB, idn2, ido2);
      while (t < t1) {
        int idn = idn1, ido = ido1;
        idn1 = idn2; ido1 = ido2;
        if (tA < t1) advance(tA, hA);
        load_ids(tA, hA, idn2, ido2);
        if (idn < 0 || ido < 0) { idn = -1; ido = -1; } // no neighbour at this offset / beyond the last site: zero rows
        const int srcId = P.swap ? ido : idn, dstId = P.swap ? idn : ido;
        { const long long c0 = P.prof ? clock64() : 0; mbar_wait(smem_u32(empty + slot), (round & 1u) ^ 1u); if (P.prof) { pwait += clock64() - c0; pstages++; } }
        const uint32_t sbase = smem_u32(sStage) + slot * stageBytes;
        if (R == 128) dw_fill_stage<128 / kDwProd>(DL, P.a, P.b, P.rowBytesA, P.rowBytesB, P.rowBytesA, P.rowBytesB, srcId, dstId, sbase, blockBytes, nBa, pw, lane);
        else dw_fill_stage<64 / kDwProd>(DL, P.a, P.b, P.rowBytesA, P.rowBytesB, P.rowBytesA, P.rowBytesB, srcId, dstId, sbase, blockBytes, nBa, pw, lane);
        cp_async_mbar_arrive_noinc(smem_u32(full + slot));
        if (++slot == (uint32_t)P.S) { slot = 0; round++; }
        t = tB; h = hB;
        tB = tA; hB = hA;
      }
    }
    if (P.prof && pw == 0 && lane == 0) { long long *q = P.prof + blockIdx.x * 8; q[0] = clock64() - pt0; q[1] = pwait; q[2] = pstages; }
  } else if (warp == kMmaWarp) {
    // ---------------- MMA issuer: both operands MN-major (bits 15, 16), M = 128, N = Cout, 32 bytes of K (= 16 bf16 / fp16, 8 tf32 positions) per instruction
    const uint32_t fmt = F16 ? 0u : BF16 ? 1u : 2u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(P.Cout >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr int kRulesPerMma = BF16 ? 16 : 8;
    const uint32_t aBlkStride16 = ((uint32_t)(nBa / nMh) * blockBytes) >> 4; // second half of M (channels 128..255): descriptor units
    uint32_t slot = 0, round = 0;
    int it = 0;
    long long mfull = 0, macc = 0;
    const long long mt0 = P.prof ? clock64() : 0;
    for (;; it++) {
      const int w = sched_take(SC, it, lane == 0);
      if (w < 0) break;
      int k, t0, t1;
      item(w, k, t0, t1);
      const int a = P.nAcc == 2 ? (it & 1) : 0, use = P.nAcc == 2 ? (it >> 1) : it;
      { const long long c0 = P.prof ? clock64() : 0; mbar_wait(smem_u32(accEmpty + a), (use & 1) ^ 1); if (P.prof) macc += clock64() - c0; }
      tc_fence_after();
      bool first = true;
      LiveTiles LT;
      LT.init(P.tileMask, k, t0, t1, tStep, lane);
      for (int t = LT.next(); t < t1; t = LT.next()) {
        for (int h = 0; h < nHalf; h++) {
          { const long long c0 = P.prof ? clock64() : 0; mbar_wait(smem_u32(full + slot), round & 1u); if (P.prof) mfull += clock64() - c0; }
          tc_fence_after();
          const uint32_t sbase = smem_u32(sStage) + slot * stageBytes;
          if (elect_one()) {
            if (R == 128) dw_issue_stage<BF16, 128 / kRulesPerMma>(sbase, blockBytes, nBa, nMh, aBlkStride16, tmemBase + (uint32_t)(a * accCols), P.Cout, idesc, first);
            else dw_issue_stage<BF16, 64 / kRulesPerMma>(sbase, blockBytes, nBa, nMh, aBlkStride16, tmemBase + (uint32_t)(a * accCols), P.Cout, idesc, first);
            tc_commit(smem_u32(empty + slot));
          }
          __syncwarp();
          first = false;
          if (++slot == (uint32_t)P.S) { slot = 0; round++; }
        }
      }
      if (elect_one()) tc_commit(smem_u32(accFull + a));
      __syncwarp();
    }
    if (P.prof && lane == 0) { long long *q = P.prof + blockIdx.x * 8; q[3] = clock64() - mt0; q[4] = mfull; q[5] = macc; }
  } else if (lane == 0) {
    // ---------------- scheduler: draws items (one beyond the end per CTA: the last CTA to do so re-zeroes the counters)
    for (int n = 0;; n++) {
      const unsigned v = atomicAdd(P.sched, 1u);
      int wi = (int)v;
      if (v >= (unsigned)nItems) {
        wi = -1;
        if (atomicAdd(P.sched + 1, 1u) == gridDim.x - 1) { P.sched[0] = 0u; P.sched[1] = 0u; }
      }
      sched_publish(SC, n, wi);
      if (wi < 0) break;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmemBase), "r"(512u) : "memory");
  }
}
// the shapes one weight-gradient launch takes: M = Cin in one or two halves of 128 rows, N = Cout, nMh x Cout TMEM columns
static bool dw_block_ok(int Cin, int Cout, int K) {
  return !((Cin % 32 != 0 && Cin > 32) || Cin > 256 || (Cin > 128 && Cin % 128 != 0) || Cout % 32 != 0 || Cout > 256 || ((Cin + 127) / 128) * Cout > 512 || K > 64);
}
// Layers wider than 256 channels on either side run as channel blocks of such shapes (launch_conv_dw_tc), from the rule lists,
// which have no filter-offset limit.
static bool dw_shape_ok(int Cin, int Cout, int K) {
  if (Cin <= 256 && Cout <= 256) return dw_block_ok(Cin, Cout, K);
  return Cin % 32 == 0 && Cout % 32 == 0 && Cin <= 1024 && Cout <= 1024 && K <= kMaxFilterVolume;
}
// whether launch_conv_dw_tc takes this shape at all (else the caller falls back to the CUDA-core kernel, which needs the fp32 rows)
bool dw_tc_ok(int Cin, int Cout, int K, int mathMode) {
  if (!half_mode(mathMode) || !tc_available()) return false;
  return dw_shape_ok(Cin, Cout, K);
}
template <bool F16>
__global__ void __launch_bounds__(256) k_from_16(const uint2 *__restrict__ x, float4 *__restrict__ y, long n4) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const uint2 v = x[i];
    if (F16) {
      const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&v.y));
      y[i] = make_float4(a.x, a.y, b.x, b.y);
    } else {
      y[i] = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xffff0000u));
    }
  }
}
// 16-bit rows in the current mode's format -> fp32 rows (exact); n a multiple of 4
int from_16(const void *x, float *y, long n, cudaStream_t s) {
  SCN_CHECK(n % 4 == 0, "16-bit -> fp32 copy needs an element count that is a multiple of 4");
  if (n && f16_copies()) k_from_16<true><<<stream_grid(n / 4, 256), 256, 0, LS(s)>>>(static_cast<const uint2 *>(x), reinterpret_cast<float4 *>(y), n / 4);
  else if (n) k_from_16<false><<<stream_grid(n / 4, 256), 256, 0, LS(s)>>>(static_cast<const uint2 *>(x), reinterpret_cast<float4 *>(y), n / 4);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
// whether launch_conv_dw_tc would run the plan-driven kernel for this shape (the caller then does not need the rule lists)
bool dw_plan_ok(int Cin, int Cout, int K, int mathMode) {
  static int planOn = -1;
  if (planOn < 0) planOn = getenv("SCN_DW_PLAN") ? atoi(getenv("SCN_DW_PLAN")) : 0;
  if (!planOn || !half_mode(mathMode) || !tc_available() || deterministic()) return false; // (its partial sums are not indexed by work item)
  return dw_block_ok(Cin, Cout, K); // (channel blocks of wider layers run from the rule lists)
}
// dW must be zero on entry.  Returns 1 when the configuration is not supported (the caller then uses the CUDA-core kernel).
// in16 / dout16: optional 16-bit copies (the mode's format) of `in` / `d_out` ([rows][Cin] / [rows][Cout], same layout) the caller already has.
int launch_conv_dw_tc(const float *in, const float *d_out, float *dW, const int2 *pairs, const int *d_off, const int *offHost, int K, long nInRows,
                      long nOutRows, int Cin, int Cout, int srcIsY, int mathMode, cudaStream_t s, const void *in16, const void *dout16,
                      const int *planNbr, const int *planOutRow, const unsigned long long *planMask, int planPos) {
  // bf16 / fp16 mode only: with TF32 operands the MN-major product came out as zeros on B200 (unresolved; tf32 mode keeps the CUDA-core kernel)
  if (!half_mode(mathMode) || !tc_available()) return 1;
  const bool bf16 = true, f16 = mathMode == kModeF16;
  if (!dw_shape_ok(Cin, Cout, K)) return 1;
  const bool wide = Cin > 256 || Cout > 256;
  const int CinP = Cin % 32 == 0 ? Cin : (Cin <= 16 ? 16 : 32); // odd narrow inputs (the 9-channel network input): bf16 rows zero-padded to 16 / 32 channels
  static int planOn = -1;
  // Measured on B470 / 6c_fpn4321 (internal numbering, 16 producer warps): level-0 32 -> 32 layers 0.45 ms with the rule lists
  // (100 % row fill, equal work items) against 0.69 ms with the plan (row fill 89 %, items of unequal cost), all 39 launches of a
  // step 2.6 against 4.2 ms -- the list kernel is the default, SCN_DW_PLAN=1 selects the plan-driven one.
  if (planOn < 0) planOn = getenv("SCN_DW_PLAN") ? atoi(getenv("SCN_DW_PLAN")) : 0;
  const bool usePlan = planOn && planNbr && planMask && planPos > 0 && !deterministic() && !wide;
  SCN_CHECK(usePlan || offHost, "weight gradient: neither a plan nor rule lists");
  const long total = usePlan ? 1 : offHost[K];
  if (total == 0) return 0;
  DwParams P;
  P.pairs = pairs; P.d_off = d_off; P.dW = dW; P.K = K; P.Cin = Cin; P.Cout = Cout; P.srcIsY = srcIsY;
  P.rowBytesA = CinP * (bf16 ? 2 : 4);
  P.rowBytesB = Cout * (bf16 ? 2 : 4);
  if (bf16) { // operand copies of both row matrices, side by side in the stream's scratch buffer
    unsigned char *scr = nullptr;
    const bool haveA = in16 && CinP == Cin, haveB = dout16 != nullptr;
    const size_t na = haveA ? 0 : (((size_t)nInRows * CinP * 2 + 255) & ~(size_t)255);
    if (!haveA || !haveB) SCN_TRY(stream_scratch(s, kScratchDw, na + (haveB ? 0 : (size_t)nOutRows * Cout * 2) + 16, (void **)&scr));
    if (haveA) ++g_counters[kCntBwdOperandReused];
    else if (CinP == Cin) SCN_TRY(to_16(in, scr, nInRows * Cin, s));
    else if (nInRows) launch_pad_rows16(in, scr, nInRows, Cin, CinP, f16, s);
    if (haveB) ++g_counters[kCntBwdOperandReused];
    else SCN_TRY(to_16(d_out, scr + na, nOutRows * Cout, s));
    P.a = haveA ? static_cast<const unsigned char *>(in16) : scr;
    P.b = haveB ? static_cast<const unsigned char *>(dout16) : scr + na;
  } else {
    P.a = reinterpret_cast<const unsigned char *>(in); P.b = reinterpret_cast<const unsigned char *>(d_out);
  }
  P.ldA = P.rowBytesA; P.ldB = P.rowBytesB; P.ldW = Cout; P.wStride = (long)Cin * Cout;
  // Channel blocks: Cin in blocks of 256 (two M halves), the rest in one block of <= 128 or 128 + the remainder; Cout in balanced
  // blocks of <= 256 (multiples of 32).  Every block is a shape dw_block_ok takes: one launch each, gathering its channel slice
  // of the same operand rows.  Layers of <= 256 x 256 are one block.
  std::vector<std::pair<int, int>> bi, bo; // (first channel, channels)
  for (int c = 0; c < Cin;) {
    const int r = Cin - c, w = !wide || r >= 256 ? std::min(r, 256) : (r <= 128 ? r : 128);
    bi.emplace_back(c, w);
    c += w;
  }
  const int nOb = wide ? cdiv(Cout, 256) : 1, units = Cout / 32;
  for (int i = 0, c = 0; i < nOb; i++) {
    const int w = wide ? 32 * (units / nOb + (i < units % nOb ? 1 : 0)) : Cout;
    bo.emplace_back(c, w);
    c += w;
  }
  const unsigned char *baseA = P.a, *baseB = P.b;
  const size_t budget = 225 * 1024 - 1024; // (the kernel also has ~1 KB of static shared memory)
  // stage shape of a block: R rules per stage, S stages, one or two TMEM accumulators
  auto shape = [&](DwParams &Q, int cinB, int coutB) {
    Q.Cin = cinB; Q.Cout = coutB;
    Q.rowBytesA = (cinB == Cin ? CinP : cinB) * 2;
    Q.rowBytesB = coutB * 2;
    const int nBlocks = std::max(Q.rowBytesA, 256) / 128 + (Q.rowBytesB + 127) / 128;
    Q.R = (size_t)nBlocks * 128 * 128 * 3 <= budget ? 128 : 64;
    const size_t stageBytes = (size_t)nBlocks * Q.R * 128;
    Q.S = (int)std::min<size_t>(4, budget / stageBytes);
    Q.nAcc = 2 * ((cinB + 127) / 128) * coutB <= 512 ? 2 : 1;
    return stageBytes;
  };
  const size_t stageBytes = shape(P, bi[0].second, bo[0].second);
  if (P.S < 2) return 1;
  if (usePlan) { // plan order (spatially coherent gathers), see conv_dw_plan_tc
    DwPlanParams Q;
    Q.a = P.a; Q.b = P.b; Q.nbr = planNbr; Q.outRow = planOutRow; Q.tileMask = planMask; Q.dW = dW;
    Q.K = K; Q.Cin = Cin; Q.Cout = Cout; Q.swap = srcIsY; Q.rowBytesA = P.rowBytesA; Q.rowBytesB = P.rowBytesB; Q.R = P.R; Q.S = P.S; Q.nAcc = P.nAcc;
    Q.nPos = planPos;
    Q.nTiles = cdiv(planPos, 128);
    static int envIpc = -1;
    if (envIpc < 0) envIpc = getenv("SCN_DW_ITEMS") ? atoi(getenv("SCN_DW_ITEMS")) : 12; // items per CTA: fine enough for the dynamic distribution to balance offsets of very different cost
    Q.itemsPerK = std::max(1, std::min(Q.nTiles, cdiv(kSMs * envIpc, K)));
    Q.chunkTiles = cdiv(Q.nTiles, Q.itemsPerK);
    Q.itemsPerK = cdiv(Q.nTiles, Q.chunkTiles);
    const size_t smemQ = (size_t)Q.S * stageBytes + 64 * 8 + 64;
    static bool attrQ = false;
    if (!attrQ) {
      SCN_CUDA(cudaFuncSetAttribute(conv_dw_plan_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
      SCN_CUDA(cudaFuncSetAttribute(conv_dw_plan_tc<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
      attrQ = true;
    }
    const int gridQ = std::min(K * Q.itemsPerK, kSMs);
    static int envProf = -1;
    if (envProf < 0) envProf = getenv("SCN_DW_PROF") ? atoi(getenv("SCN_DW_PROF")) : 0;
    Q.prof = nullptr;
    if (envProf) { SCN_CUDA(cudaMalloc((void **)&Q.prof, kSMs * 8 * 8)); SCN_CUDA(cudaMemsetAsync(Q.prof, 0, kSMs * 8 * 8, s)); }
    SCN_TRY(sched_counters(s, &Q.sched));
    ++g_counters[kCntFloatAtomic];
    if (f16) { ++g_counters[kCntF16Launch]; conv_dw_plan_tc<true, true><<<gridQ, 32 * (6 + kDwProd), smemQ, LS(s)>>>(Q); }
    else conv_dw_plan_tc<true><<<gridQ, 32 * (6 + kDwProd), smemQ, LS(s)>>>(Q);
    SCN_CUDA(cudaGetLastError());
    if (envProf) { // developer aid: per-role cycle counters, mean and max over the CTAs
      static long long h[kSMs * 8];
      SCN_CUDA(cudaMemcpyAsync(h, Q.prof, sizeof h, cudaMemcpyDeviceToHost, s));
      SCN_CUDA(cudaStreamSynchronize(s));
      double mean[8] = {0}, mx[8] = {0};
      for (int b = 0; b < gridQ; b++) for (int i = 0; i < 8; i++) { mean[i] += (double)h[b * 8 + i] / gridQ; mx[i] = std::max(mx[i], (double)h[b * 8 + i]); }
      fprintf(stderr, "[dwprof] K=%d Cin=%d Cout=%d tiles=%d items/K=%d R=%d S=%d | producer total %.0f (max %.0f) wait-empty %.0f stages %.0f (max %.0f) | mma total %.0f wait-full %.0f wait-acc %.0f\n",
              K, Cin, Cout, Q.nTiles, Q.itemsPerK, Q.R, Q.S, mean[0], mx[0], mean[1], mean[2], mx[2], mean[3], mean[4], mean[5]);
      cudaFree(Q.prof);
    }
    ++g_counters[kCntDwPlanLaunch];
    return 0;
  }
  // parts per list: ~4K rules each on the large levels (the rows of all offsets of the parts in flight then fit in L2), at least
  // ~3 items per SM where the lists are long enough, never parts of fewer than 4 stages
  static int envPart = -1;
  if (envPart < 0) envPart = getenv("SCN_DW_PART") ? atoi(getenv("SCN_DW_PART")) : 4096;
  const long avgLen = std::max<long>(1, total / K);
  long nC = std::max<long>(1, avgLen / envPart);
  if (K * nC < 3 * kSMs) nC = std::max<long>(nC, std::min<long>(cdiv(3 * kSMs, K), std::max<long>(1, avgLen / (4 * P.R))));
  P.nC = (int)std::min<long>(nC, 4096);
  P.part = nullptr;
  if (deterministic()) { // one dW-sized slot per work item, at most kDetDwBytes in all (fewer, longer parts beyond that)
    constexpr size_t kDetDwBytes = 256u << 20;
    const size_t perItem = (size_t)Cin * Cout * 4;
    P.nC = (int)std::max<size_t>(1, std::min<size_t>((size_t)P.nC, kDetDwBytes / (perItem * K)));
    // (a wide layer with one part per list: item k is the only writer of dW[k] -- its plain stores go to dW, no workspace)
    if (wide && P.nC == 1) P.part = dW;
    else SCN_TRY(det_scratch(s, (size_t)K * P.nC * perItem, (void **)&P.part));
  } else {
    g_counters[kCntFloatAtomic] += (long)(bi.size() * bo.size()); // (one per launch)
  }
  const long nItems = (long)K * P.nC;
  static bool attr = false;
  if (!attr) {
    SCN_CUDA(cudaFuncSetAttribute(conv_dw_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    SCN_CUDA(cudaFuncSetAttribute(conv_dw_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    SCN_CUDA(cudaFuncSetAttribute(conv_dw_tc<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
    attr = true;
  }
  const int grid = (int)std::min<long>(nItems, kSMs);
  // every block with the same parts per list: in deterministic mode they all fill the one [nC][K][Cin][Cout] workspace
  for (const auto &ib : bi)
    for (const auto &ob : bo) {
      DwParams Q = P;
      const size_t sb = shape(Q, ib.second, ob.second);
      SCN_CHECK(Q.S >= 2, "weight gradient: channel block does not fit in shared memory");
      Q.a = baseA + (size_t)ib.first * 2; Q.b = baseB + (size_t)ob.first * 2;
      Q.dW = dW + (size_t)ib.first * Cout + ob.first;
      if (P.part) Q.part = P.part + (size_t)ib.first * Cout + ob.first;
      const size_t smemBytes = (size_t)Q.S * sb + 64 * 8 + 64;
      if (f16) { ++g_counters[kCntF16Launch]; conv_dw_tc<true, true><<<grid, 32 * (5 + kDwProd), smemBytes, LS(s)>>>(Q); }
      else if (bf16) conv_dw_tc<true><<<grid, 32 * (5 + kDwProd), smemBytes, LS(s)>>>(Q);
      else conv_dw_tc<false><<<grid, 32 * (5 + kDwProd), smemBytes, LS(s)>>>(Q);
      SCN_CUDA(cudaGetLastError());
    }
  if (P.part && P.part != dW) SCN_TRY(ordered_sum(P.part, P.nC, (long)K * Cin * Cout, dW, s)); // item c K + k = part c of list k: rows [nC][K][Cin][Cout]
  return 0;
}

// frees the cached weight operand images and the per-stream scratch buffers (the caller has synchronised the device) -> bytes released
long release_conv_caches() {
  long freed = 0;
  {
    std::lock_guard<std::mutex> lk(g_wimg_mu);
    for (auto &kv : g_wimg) { cudaFree(kv.second.img); cudaEventDestroy(kv.second.ready); freed += (long)kv.second.bytes; }
    g_wimg.clear();
    g_wimg_bytes = 0;
  }
  {
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    for (auto &kv : g_scratch) if (kv.second.first) { cudaFree(kv.second.first); freed += (long)kv.second.second; }
    g_scratch.clear();
  }
  return freed;
}

} // namespace scn
