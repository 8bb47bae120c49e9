// fp32 CUDA-core gather-GEMM kernels: the exact-fp32 path (tolerance anchor for the tensor-core
// path, and the only path for channel counts the tcgen05 kernel does not take, e.g. Cin = 9).
//
//  * conv_plan_simt : output-stationary.  A CTA owns 64 output sites (in spatial order) x 64 output
//    channels and loops over the filter offsets that have at least one neighbour inside the tile,
//    gathering input rows by the plan's neighbour table.  One store per output element, no
//    read-modify-write, no atomics (replaces dConvolution_KMxKN_forwardA/B + RULEBOOKITERATOR,
//    SCN/CUDA/Convolution.cu:57-203, RuleBookIterator.h:15-32).
//  * conv_list_simt : rule-list driven (gather rows by pairs[i].src, write rows pairs[i].dst) for
//    deconvolution, where every fine row has one parent (SCN/CUDA/Deconvolution.cu).
#include "conv.cuh"

namespace scn {

constexpr int TM = 64, TN = 64, KC = 16, APAD = 4;

template <bool VEC>
__device__ __forceinline__ void load_a_chunk(const float *__restrict__ in, int row, int Cin, int c0, int tid, float (*A_s)[TM + APAD]) {
  const int rr = tid >> 2, c4 = (tid & 3) * 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (row >= 0) {
    const float *src = in + (long)row * Cin + c0 + c4;
    if (VEC) {
      if (c0 + c4 < Cin) { float4 t = __ldg(reinterpret_cast<const float4 *>(src)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) if (c0 + c4 + j < Cin) v[j] = __ldg(src + j);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; j++) A_s[c4 + j][rr] = v[j];
}
template <bool VEC>
__device__ __forceinline__ void load_b_chunk(const float *__restrict__ Wk, int Cin, int Cout, int c0, int n0, int tid, float (*B_s)[TN]) {
  const int kk = tid >> 4, n4 = (tid & 15) * 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (c0 + kk < Cin) {
    const float *src = Wk + (long)(c0 + kk) * Cout + n0 + n4;
    if (VEC) {
      if (n0 + n4 < Cout) { float4 t = __ldg(reinterpret_cast<const float4 *>(src)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) if (n0 + n4 + j < Cout) v[j] = __ldg(src + j);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; j++) B_s[kk][n4 + j] = v[j];
}
__device__ __forceinline__ void mma_chunk(const float (*A_s)[TM + APAD], const float (*B_s)[TN], int tx, int ty, float acc[4][4]) {
#pragma unroll
  for (int kk = 0; kk < KC; kk++) {
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; i++) a[i] = A_s[kk][ty * 4 + i];
    float4 bv = *reinterpret_cast<const float4 *>(&B_s[kk][tx * 4]);
    b[0] = bv.x; b[1] = bv.y; b[2] = bv.z; b[3] = bv.w;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

// WIDE: a plan of more than 64 filter offsets (chunk-major, nbr_index_wide); one launch still sums all offsets in order
template <bool VEC, bool WIDE = false>
__global__ void __launch_bounds__(256) conv_plan_simt(const float *__restrict__ in, float *__restrict__ out, const float *__restrict__ W,
                                                      const int *__restrict__ nbr, const int *__restrict__ outRow, int nOut, int K, int Cin, int Cout,
                                                      const float *__restrict__ bias) {
  __shared__ __align__(16) float A_s[KC][TM + APAD];
  __shared__ __align__(16) float B_s[KC][TN];
  __shared__ int s_ids[TM];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int p0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  for (int k = 0; k < K; k++) {
    int id = -1;
    if (tid < TM && p0 + tid < nOut)
      id = nbr ? __ldg(nbr + (WIDE ? nbr_index_wide(p0 + tid, k, K, plan_padded(nOut)) : nbr_index(p0 + tid, k, K))) : p0 + tid; // no plan: dense rows (NetworkInNetwork)
    __syncthreads(); // previous offset's readers of s_ids / tiles are done
    if (tid < TM) s_ids[tid] = id;
    if (!__syncthreads_or(id >= 0)) continue;
    const int myrow = s_ids[tid >> 2];
    const float *Wk = W + (long)k * Cin * Cout;
    for (int c0 = 0; c0 < Cin; c0 += KC) {
      load_a_chunk<VEC>(in, myrow, Cin, c0, tid, A_s);
      load_b_chunk<VEC>(Wk, Cin, Cout, c0, n0, tid, B_s);
      __syncthreads();
      mma_chunk(A_s, B_s, tx, ty, acc);
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int p = p0 + ty * 4 + i;
    if (p >= nOut) continue;
    float *dst = out + (long)(outRow ? __ldg(outRow + p) : p) * Cout + n0 + tx * 4;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      int c = n0 + tx * 4 + j;
      if (c < Cout) dst[j] = acc[i][j] + (bias ? __ldg(bias + c) : 0.f);
    }
  }
}

// conv_plan_simt2: the same product with a larger register tile and a software pipeline.  A CTA owns one plan tile (128 output
// sites) x TN2 output channels; a thread holds 8 sites x (TN2 / 16) channels.  The (filter offset, 16-channel chunk) steps of ALL
// live offsets form one sequence: while the FMAs of step s run out of one shared-memory buffer, the rows and weights of step
// s + 1 are already on their way into registers and are stored into the other buffer afterwards -- one barrier per step, no bubble
// at the offset boundaries (32-channel layers have only two chunks per offset).  The neighbour ids of the whole tile (K x 128)
// are read once, coalesced, into shared memory; offsets without a neighbour in the tile are skipped.
// Measured on B470 (fp32 mode): dominant layer 11.3 -> 10.9 ms (32 TFLOP/s = 43 % of the fp32 FMA peak), whole forward 34.2 -> 32.7 ms:
// the exact path stays bound by its 512-byte row gathers through ordinary loads, not by the FMA issue rate.
constexpr int TM2 = 128, KC2 = 16, APAD2 = 4, KMAX2 = 32;
template <int TN2>
__global__ void __launch_bounds__(256) conv_plan_simt2(const float *__restrict__ in, float *__restrict__ out, const float *__restrict__ W,
                                                       const int *__restrict__ nbr, const int *__restrict__ outRow, int nOut, int K, int Cin, int Cout,
                                                       const float *__restrict__ bias) {
  constexpr int CPT = TN2 / 16; // output channels per thread (4 or 2)
  __shared__ __align__(16) float A_s[2][KC2][TM2 + APAD2];
  __shared__ __align__(16) float B_s[2][KC2][TN2];
  __shared__ int s_ids[KMAX2][TM2];
  __shared__ int s_live[KMAX2 + 1]; // live offsets, s_live[KMAX2] = their number
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
  const long tile = blockIdx.x;
  const int n0 = blockIdx.y * TN2;
  // ids of the tile: nbr[(tile K + k) 128 + r], contiguous
  unsigned liveBits = 0; // (warp w collects offsets w, w + 8, ...)
  for (int k = warp; k < K; k += 8) {
    bool any = false;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int id = __ldg(nbr + (tile * K + k) * 128 + q * 32 + lane);
      s_ids[k][q * 32 + lane] = id;
      any |= id >= 0;
    }
    if (__any_sync(0xffffffffu, any)) liveBits |= 1u << k;
  }
  if (tid == 0) s_live[KMAX2] = 0;
  __syncthreads();
  if (lane == 0 && liveBits) atomicOr(reinterpret_cast<unsigned *>(&s_live[KMAX2]), liveBits); // (bit set first, compacted below)
  __syncthreads();
  if (tid == 0) {
    unsigned bits = (unsigned)s_live[KMAX2];
    int n = 0;
    while (bits) { s_live[n++] = __ffs(bits) - 1; bits &= bits - 1; }
    s_live[KMAX2] = n;
  }
  __syncthreads();
  const int nLive = s_live[KMAX2], nChunks = Cin / KC2, nSteps = nLive * nChunks;
  float acc[8][CPT];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < CPT; j++) acc[i][j] = 0.f;
  // loader roles: A -- thread t reads 8 consecutive channels of row t / 2; B -- thread t reads 4 consecutive output channels of input channel t / (TN2 / 4)
  const int aRow = tid >> 1, aC = (tid & 1) * 8;
  constexpr int BT = KC2 * TN2 / 4; // threads that load B (256 for TN2 = 64, 128 for TN2 = 32)
  const int bK = tid / (TN2 / 4), bN = (tid % (TN2 / 4)) * 4;
  float4 ra0, ra1, rb;
  auto fetch = [&](int step) {
    const int k = s_live[step / nChunks], c0 = (step % nChunks) * KC2;
    const int id = s_ids[k][aRow];
    ra0 = ra1 = rb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (id >= 0) {
      const float4 *src = reinterpret_cast<const float4 *>(in + (long)id * Cin + c0 + aC);
      ra0 = __ldg(src);
      ra1 = __ldg(src + 1);
    }
    if (tid < BT && n0 + bN < Cout) rb = __ldg(reinterpret_cast<const float4 *>(W + ((long)k * Cin + c0 + bK) * Cout + n0 + bN));
  };
  auto stash = [&](int buf) {
    A_s[buf][aC + 0][aRow] = ra0.x; A_s[buf][aC + 1][aRow] = ra0.y; A_s[buf][aC + 2][aRow] = ra0.z; A_s[buf][aC + 3][aRow] = ra0.w;
    A_s[buf][aC + 4][aRow] = ra1.x; A_s[buf][aC + 5][aRow] = ra1.y; A_s[buf][aC + 6][aRow] = ra1.z; A_s[buf][aC + 7][aRow] = ra1.w;
    if (tid < BT) *reinterpret_cast<float4 *>(&B_s[buf][bK][bN]) = rb;
  };
  if (nSteps > 0) {
    fetch(0);
    stash(0);
    __syncthreads();
    for (int step = 0; step < nSteps; step++) {
      const int buf = step & 1;
      if (step + 1 < nSteps) fetch(step + 1);
#pragma unroll
      for (int kk = 0; kk < KC2; kk++) {
        const float4 a0 = *reinterpret_cast<const float4 *>(&A_s[buf][kk][ty * 8]), a1 = *reinterpret_cast<const float4 *>(&A_s[buf][kk][ty * 8 + 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float b[CPT];
        if (CPT == 4) { const float4 bv = *reinterpret_cast<const float4 *>(&B_s[buf][kk][tx * 4]); b[0] = bv.x; b[1] = bv.y; b[2] = bv.z; b[3] = bv.w; }
        else { const float2 bv = *reinterpret_cast<const float2 *>(&B_s[buf][kk][tx * 2]); b[0] = bv.x; b[1] = bv.y; }
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
          for (int j = 0; j < CPT; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      if (step + 1 < nSteps) stash(buf ^ 1); // (the other buffer's readers passed the barrier at the end of the previous step)
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const long p = tile * TM2 + ty * 8 + i;
    if (p >= nOut) continue;
    float *dst = out + (long)(outRow ? __ldg(outRow + p) : p) * Cout + n0 + tx * CPT;
#pragma unroll
    for (int j = 0; j < CPT; j++) {
      const int c = n0 + tx * CPT + j;
      if (c < Cout) dst[j] = acc[i][j] + (bias ? __ldg(bias + c) : 0.f);
    }
  }
}

// Rule-list driven: tile = 64 consecutive pairs of one list.
template <bool VEC>
__global__ void __launch_bounds__(256) conv_list_simt(const float *__restrict__ in, float *__restrict__ out, const float *__restrict__ W,
                                                      const int2 *__restrict__ pairs, const int *__restrict__ off, int K, int Cin, int Cout,
                                                      int srcIsY, int accumulate, int onlyList) {
  __shared__ __align__(16) float A_s[KC][TM + APAD];
  __shared__ __align__(16) float B_s[KC][TN];
  __shared__ int s_src[TM], s_dst[TM];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  // locate (list, first pair) of this tile
  int t = blockIdx.x, L = 0, start = 0, len = 0;
  if (onlyList >= 0) { L = onlyList; start = off[L]; len = off[L + 1] - start; }
  else {
    for (L = 0; L < K; L++) {
      start = off[L]; len = off[L + 1] - start;
      int tiles = (len + TM - 1) / TM;
      if (t < tiles) break;
      t -= tiles;
    }
    if (L == K) return;
  }
  const int i0 = t * TM, n0 = blockIdx.y * TN;
  if (tid < TM) {
    int2 pr = make_int2(-1, -1);
    if (i0 + tid < len) pr = __ldg(pairs + start + i0 + tid);
    s_src[tid] = srcIsY ? pr.y : pr.x;
    s_dst[tid] = srcIsY ? pr.x : pr.y;
  }
  __syncthreads();
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  const int myrow = s_src[tid >> 2];
  const float *Wk = W + (long)L * Cin * Cout;
  for (int c0 = 0; c0 < Cin; c0 += KC) {
    load_a_chunk<VEC>(in, myrow, Cin, c0, tid, A_s);
    load_b_chunk<VEC>(Wk, Cin, Cout, c0, n0, tid, B_s);
    __syncthreads();
    mma_chunk(A_s, B_s, tx, ty, acc);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int d = s_dst[ty * 4 + i];
    if (d < 0) continue;
    float *dst = out + (long)d * Cout + n0 + tx * 4;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      int c = n0 + tx * 4 + j;
      if (c < Cout) dst[j] = accumulate ? dst[j] + acc[i][j] : acc[i][j];
    }
  }
}

int launch_conv_plan_simt(const float *in, float *out, const float *W, const int *nbr, const int *outRow, int nOut, int K, int Cin, int Cout,
                          const float *bias, cudaStream_t s) {
  if (nOut == 0) return 0;
  ++g_counters[kCntSimtLaunch];
  static int v2 = -1;
  if (v2 < 0) v2 = getenv("SCN_SIMT2") ? atoi(getenv("SCN_SIMT2")) : 1; // developer switch: 0 = the 64 x 64 kernel always
  if (v2 && nbr && K <= KMAX2 && Cin % KC2 == 0 && Cout % 4 == 0) { // plan tiles of 128 sites, 16-channel chunks, vector stores
    if (Cout <= 32) conv_plan_simt2<32><<<dim3(cdiv(nOut, TM2), cdiv(Cout, 32)), 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
    else conv_plan_simt2<64><<<dim3(cdiv(nOut, TM2), cdiv(Cout, 64)), 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
    SCN_CUDA(cudaGetLastError());
    return 0;
  }
  dim3 grid(cdiv(nOut, TM), cdiv(Cout, TN));
  if (K > 64 && Cin % 4 == 0 && Cout % 4 == 0)
    conv_plan_simt<true, true><<<grid, 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
  else if (K > 64)
    conv_plan_simt<false, true><<<grid, 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
  else if (Cin % 4 == 0 && Cout % 4 == 0)
    conv_plan_simt<true><<<grid, 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
  else
    conv_plan_simt<false><<<grid, 256, 0, LS(s)>>>(in, out, W, nbr, outRow, nOut, K, Cin, Cout, bias);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// offHost: list offsets on the host (K+1).  singleParent: every dst row occurs in exactly one rule.
int launch_conv_list_simt(const float *in, float *out, const float *W, const int2 *pairs, const int *d_off, const int *offHost, int K, int Cin,
                          int Cout, int srcIsY, int singlePass, cudaStream_t s) {
  const bool vec = Cin % 4 == 0 && Cout % 4 == 0;
  ++g_counters[kCntSimtLaunch];
  if (singlePass) {
    long tiles = 0;
    for (int L = 0; L < K; L++) tiles += cdiv(offHost[L + 1] - offHost[L], TM);
    if (!tiles) return 0;
    dim3 grid((unsigned)tiles, cdiv(Cout, TN));
    if (vec) conv_list_simt<true><<<grid, 256, 0, LS(s)>>>(in, out, W, pairs, d_off, K, Cin, Cout, srcIsY, 0, -1);
    else conv_list_simt<false><<<grid, 256, 0, LS(s)>>>(in, out, W, pairs, d_off, K, Cin, Cout, srcIsY, 0, -1);
  } else { // a dst row may occur once per list: lists run back to back, read-modify-write
    for (int L = 0; L < K; L++) {
      int len = offHost[L + 1] - offHost[L];
      if (!len) continue;
      dim3 grid(cdiv(len, TM), cdiv(Cout, TN));
      if (vec) conv_list_simt<true><<<grid, 256, 0, LS(s)>>>(in, out, W, pairs, d_off, K, Cin, Cout, srcIsY, 1, L);
      else conv_list_simt<false><<<grid, 256, 0, LS(s)>>>(in, out, W, pairs, d_off, K, Cin, Cout, srcIsY, 1, L);
    }
  }
  SCN_CUDA(cudaGetLastError());
  return 0;
}

} // namespace scn
