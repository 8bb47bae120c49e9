// Row-wise (HBM-bound) kernels: BatchNorm(+leaky ReLU) forward/backward, InputLayer
// forward/backward, feature-plane addition.  All stream rows with 16-byte accesses and size
// their grids as multiples of the 148 SMs.
//
// Replaces BatchNormalization_f_train/f_test/b (SCN/CUDA/BatchNormalization.cu:14-198, which run
// on <= 16 CTAs) and InputLayer_fp_/bp_ (SCN/CUDA/IOLayers.cu:14-58).
#include "common.cuh"
#include <cuda_bf16.h>

namespace scn {

// mode 0: train   -- BatchNormalization_ForwardPass train branch (SCN/CPU/BatchNormalization.cpp:19-40):
//                    biased variance for normalisation, running stats updated with unbiased variance.
// mode 1: eval with given running stats (:41-46).
// mode 2: eval, track_running_stats=False -- sparseconvnet/batchNormalization.py:51-56: mean(0) and the
//                    UNBIASED var(0) of this input stand in for the running stats.
// (sum, sumsq) -> saveMean / saveInvStd and the fused scale / shift of  y = x*scale + shift.
struct BnFin {
  long n; int C, mode; float eps, momentum;
  float *saveMean, *saveInvStd, *runningMean, *runningVar;
  const float *weight, *bias;
  float *scale, *shift;
};
__device__ __forceinline__ void bn_finalize_channel(const BnFin &F, int c, double sum, double sumsq) {
  float mean, invstd;
  if (F.mode == 1) {
    mean = F.runningMean[c];
    invstd = powf(F.runningVar[c] + F.eps, -0.5f);
  } else {
    double m = sum / (double)F.n;
    double ss = sumsq - m * m * (double)F.n; // sum of squared deviations
    if (ss < 0) ss = 0;
    mean = (float)m;
    if (F.mode == 0) {
      F.runningMean[c] = F.momentum * F.runningMean[c] + (1 - F.momentum) * mean;
      F.runningVar[c] = F.momentum * F.runningVar[c] + (1 - F.momentum) * (float)(ss / (double)(F.n - 1));
      invstd = powf((float)(ss / (double)F.n) + F.eps, -0.5f);
    } else {
      invstd = powf((float)(ss / (double)(F.n - 1)) + F.eps, -0.5f);
    }
  }
  F.saveMean[c] = mean;
  F.saveInvStd[c] = invstd;
  float w = invstd * (F.weight ? F.weight[c] : 1.f);
  F.scale[c] = w;
  F.shift[c] = -mean * w + (F.bias ? F.bias[c] : 0.f);
}
// ------------------------------------------------------------------ ordered sums (deterministic mode)
// Column j of a [nPart][width] matrix of partial sums: 32 row lanes each add the rows lane, lane + 32, ... in ascending order, then
// one thread adds the 32 lane sums in lane order.  The order depends on nPart and width only, never on the scheduling.
template <class T>
__global__ void __launch_bounds__(1024) k_ordered_sum(const T *__restrict__ part, int nPart, long width, T *__restrict__ out, long seg, long segStride) {
  __shared__ double red[32][33];
  const long j = (long)blockIdx.x * 32 + threadIdx.x;
  double a = 0.0;
  if (j < width)
    for (int p = threadIdx.y; p < nPart; p += 32) a += (double)part[(long)p * width + j];
  red[threadIdx.y][threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.y == 0 && j < width) {
    double t = 0.0;
    for (int l = 0; l < 32; l++) t += red[l][threadIdx.x];
    out[seg > 0 ? (j / seg) * segStride + j % seg : j] = (T)t;
  }
}
template <class T>
int ordered_sum(const T *part, int nPart, long width, T *out, cudaStream_t s, long seg, long segStride) {
  if (width <= 0) return 0;
  k_ordered_sum<T><<<cdiv(width, 32), dim3(32, 32), 0, LS(s)>>>(part, nPart, width, out, seg, segStride);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
template int ordered_sum<float>(const float *, int, long, float *, cudaStream_t, long, long);
template int ordered_sum<double>(const double *, int, long, double *, cudaStream_t, long, long);

// ------------------------------------------------------------------ BN statistics
// stats[0..C) = sum x, stats[C..2C) = sum x^2 (or sum of (x-shift)^2 terms), in double.
// Each thread owns one float4 column group and strides over rows; per-CTA partials are reduced
// in shared memory and added with one double atomic per channel per CTA.
// The CTA that finishes last (ticket) turns the sums into scale / shift and re-zeroes sums and ticket:
// statistics + finalize are one launch.
// part (deterministic mode): the CTA's sums go to row blockIdx.x of part [grid][2][C] instead; ordered_sum + k_bn_finalize follow.
__global__ void __launch_bounds__(256) k_bn_stats(const float *__restrict__ x, long n, int C, int rowsPerCta, double *__restrict__ stats,
                                                  unsigned *ticket, BnFin F, double *__restrict__ part) {
  extern __shared__ float s_red[]; // [2][256][4]
  const int cv = C >> 2;           // float4 groups per row
  const int tid = threadIdx.x;
  const int lanesPerRow = cv;      // cv <= 256
  const int rowLanes = 256 / lanesPerRow;
  const int cg = tid % lanesPerRow, rl = tid / lanesPerRow;
  float4 s = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
  const long r0 = (long)blockIdx.x * rowsPerCta;
  const long r1 = min(n, r0 + rowsPerCta);
  if (rl < rowLanes) {
    long r = r0 + rl;
    for (; r + 3l * rowLanes < r1; r += 4l * rowLanes) { // 4 independent 16-byte loads in flight per thread
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) v[u] = __ldg(reinterpret_cast<const float4 *>(x + (r + (long)u * rowLanes) * C) + cg);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w;
        q.x = fmaf(v[u].x, v[u].x, q.x); q.y = fmaf(v[u].y, v[u].y, q.y); q.z = fmaf(v[u].z, v[u].z, q.z); q.w = fmaf(v[u].w, v[u].w, q.w);
      }
    }
    for (; r < r1; r += rowLanes) {
      float4 v = __ldg(reinterpret_cast<const float4 *>(x + r * C) + cg);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
    }
  }
  float4 *S = reinterpret_cast<float4 *>(s_red), *Q = S + 256;
  S[tid] = s; Q[tid] = q;
  __syncthreads();
  if (tid < lanesPerRow) {
    double a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
    for (int l = 0; l < rowLanes; l++) {
      float4 u = S[l * lanesPerRow + tid], w = Q[l * lanesPerRow + tid];
      a[0] += u.x; a[1] += u.y; a[2] += u.z; a[3] += u.w;
      b[0] += w.x; b[1] += w.y; b[2] += w.z; b[3] += w.w;
    }
    if (part) {
      double *row = part + (size_t)blockIdx.x * 2 * C;
#pragma unroll
      for (int j = 0; j < 4; j++) { row[tid * 4 + j] = a[j]; row[C + tid * 4 + j] = b[j]; }
    } else {
      double *rep = stats + (size_t)(blockIdx.x % kBnReplicas) * 2 * kBnMaxC; // same-address double atomics cost ~45 ns each: spread them
#pragma unroll
      for (int j = 0; j < 4; j++) {
        atomicAdd(rep + tid * 4 + j, a[j]);
        atomicAdd(rep + C + tid * 4 + j, b[j]);
      }
    }
  }
  if (part) return; // (uniform over the grid)
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence();
    volatile double *vs = stats;
    for (int c = tid; c < C; c += 256) {
      double a = 0, b = 0;
      for (int r = 0; r < kBnReplicas; r++) {
        volatile double *vr = vs + (size_t)r * 2 * kBnMaxC;
        a += vr[c]; b += vr[C + c];
        vr[c] = 0.0; vr[C + c] = 0.0;
      }
      bn_finalize_channel(F, c, a, b);
    }
    if (tid == 0) *ticket = 0u;
  }
}
// One launch for small inputs: CTA b owns channels [32 b, 32 b + 32); statistics, scale / shift and the
// normalised output (the rows come back out of L1/L2 for the second pass).
__global__ void __launch_bounds__(256) k_bn_small(const float *__restrict__ x, float *__restrict__ y, int n, int C, BnFin F, float leak, void *__restrict__ y16) {
  __shared__ float4 S[256], Q[256];
  __shared__ float sScale[32], sShift[32];
  pdl_launch_dependents();
  pdl_wait();
  const int tid = threadIdx.x, cgl = tid & 7, rl = tid >> 3; // 8 float4 column groups x 32 row lanes
  const int cg = blockIdx.x * 8 + cgl, cv = C >> 2;
  const bool live = cg < cv;
  float4 s = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
  if (live && F.mode != 1)
    for (int r = rl; r < n; r += 32) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(x + (long)r * C) + cg);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
    }
  S[tid] = s; Q[tid] = q;
  __syncthreads();
  if (tid < 32) { // one thread per channel of this CTA
    const int c = blockIdx.x * 32 + tid, g = tid >> 2, j = tid & 3;
    if (c < C) {
      double a = 0, b = 0;
      for (int l = 0; l < 32; l++) {
        const float4 u = S[l * 8 + g], w = Q[l * 8 + g];
        a += j == 0 ? u.x : j == 1 ? u.y : j == 2 ? u.z : u.w;
        b += j == 0 ? w.x : j == 1 ? w.y : j == 2 ? w.z : w.w;
      }
      bn_finalize_channel(F, c, a, b);
      sScale[tid] = F.scale[c];
      sShift[tid] = F.shift[c];
    }
  }
  __syncthreads();
  if (!live) return;
  const float4 a = make_float4(sScale[cgl * 4], sScale[cgl * 4 + 1], sScale[cgl * 4 + 2], sScale[cgl * 4 + 3]);
  const float4 b = make_float4(sShift[cgl * 4], sShift[cgl * 4 + 1], sShift[cgl * 4 + 2], sShift[cgl * 4 + 3]);
  for (int r = rl; r < n; r += 32) {
    const long i = (long)r * cv + cg;
    const float4 v = __ldg(reinterpret_cast<const float4 *>(x) + i);
    float4 o;
    o.x = fmaf(v.x, a.x, b.x); o.y = fmaf(v.y, a.y, b.y); o.z = fmaf(v.z, a.z, b.z); o.w = fmaf(v.w, a.w, b.w);
    o.x = o.x > 0 ? o.x : o.x * leak; o.y = o.y > 0 ? o.y : o.y * leak; o.z = o.z > 0 ? o.z : o.z * leak; o.w = o.w > 0 ? o.w : o.w * leak;
    reinterpret_cast<float4 *>(y)[i] = o;
    if (y16) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
      uint2 pk;
      pk.x = *reinterpret_cast<unsigned int *>(&lo);
      pk.y = *reinterpret_cast<unsigned int *>(&hi);
      reinterpret_cast<uint2 *>(y16)[i] = pk;
    }
  }
}
// scalar fallback for C % 4 != 0 (C <= 256)
__global__ void __launch_bounds__(256) k_bn_stats_scalar(const float *__restrict__ x, long n, int C, int rowsPerCta, double *__restrict__ stats,
                                                         double *__restrict__ part) {
  __shared__ float S[256], Q[256];
  const int tid = threadIdx.x;
  const int rowLanes = 256 / C;
  const int c = tid % C, rl = tid / C;
  float s = 0.f, q = 0.f;
  const long r0 = (long)blockIdx.x * rowsPerCta, r1 = min(n, r0 + rowsPerCta);
  if (rl < rowLanes)
    for (long r = r0 + rl; r < r1; r += rowLanes) { float v = __ldg(x + r * C + c); s += v; q = fmaf(v, v, q); }
  S[tid] = s; Q[tid] = q;
  __syncthreads();
  if (tid < C) {
    double a = 0, b = 0;
    for (int l = 0; l < rowLanes; l++) { a += S[l * C + tid]; b += Q[l * C + tid]; }
    if (part) { part[(size_t)blockIdx.x * 2 * C + tid] = a; part[(size_t)blockIdx.x * 2 * C + C + tid] = b; }
    else { atomicAdd(stats + tid, a); atomicAdd(stats + C + tid, b); }
  }
}

// standalone finalize: eval with running statistics (no sums needed) and the scalar-statistics path
__global__ void k_bn_finalize(double *__restrict__ stats, BnFin F) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= F.C) return;
  double a = 0, b = 0;
  if (F.mode != 1) { a = stats[c]; b = stats[F.C + c]; stats[c] = 0.0; stats[F.C + c] = 0.0; }
  bn_finalize_channel(F, c, a, b);
}

// y = leaky(x*scale + shift)   (:53-61)
// y16 (optional): the same values rounded to bf16, the gather operand of a following bf16 convolution
__device__ __forceinline__ void store_bf16x4(void *base, long i, float4 o) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
  uint2 pk;
  pk.x = *reinterpret_cast<unsigned int *>(&lo);
  pk.y = *reinterpret_cast<unsigned int *>(&hi);
  reinterpret_cast<uint2 *>(base)[i] = pk;
}
__global__ void __launch_bounds__(256) k_bn_apply(const float *__restrict__ x, float *__restrict__ y, long total4, int cv, const float *__restrict__ scale,
                                                  const float *__restrict__ shift, float leak, void *__restrict__ y16) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total4; i += (long)gridDim.x * blockDim.x) {
    int cg = (int)(i % cv);
    float4 v = __ldg(reinterpret_cast<const float4 *>(x) + i);
    float4 a = __ldg(reinterpret_cast<const float4 *>(scale) + cg), b = __ldg(reinterpret_cast<const float4 *>(shift) + cg);
    float4 o;
    o.x = fmaf(v.x, a.x, b.x); o.y = fmaf(v.y, a.y, b.y); o.z = fmaf(v.z, a.z, b.z); o.w = fmaf(v.w, a.w, b.w);
    o.x = o.x > 0 ? o.x : o.x * leak; o.y = o.y > 0 ? o.y : o.y * leak; o.z = o.z > 0 ? o.z : o.z * leak; o.w = o.w > 0 ? o.w : o.w * leak;
    reinterpret_cast<float4 *>(y)[i] = o;
    if (y16) store_bf16x4(y16, i, o);
  }
}
__global__ void __launch_bounds__(256) k_bn_apply_scalar(const float *__restrict__ x, float *__restrict__ y, long total, int C, const float *__restrict__ scale,
                                                         const float *__restrict__ shift, float leak) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    float o = fmaf(__ldg(x + i), scale[c], shift[c]);
    y[i] = o > 0 ? o : o * leak;
  }
}

// y = leaky(x*scale + shift) with scale / shift derived in the kernel's prologue from per-channel sums that the
// PRODUCER of x accumulated in its epilogue (conv_plan_tc, P.stats): the statistics pass over x disappears.
// sums: [kBnReplicas][2][kFusedStatsC] doubles.  Block 0 also writes saveMean / saveInvStd and (train mode) the
// running statistics, exactly once.
__global__ void __launch_bounds__(256) k_bn_apply_sums(const float *__restrict__ x, float *__restrict__ y, long total4, int cv, const double *__restrict__ sums,
                                                       BnFin F, float leak, void *__restrict__ y16) {
  __shared__ __align__(16) float sScale[kFusedStatsC], sShift[kFusedStatsC];
  pdl_launch_dependents();
  pdl_wait(); // (the sums come from the producing convolution's epilogue)
  for (int c = threadIdx.x; c < F.C; c += 256) {
    double a = 0, b = 0;
    for (int r = 0; r < kBnReplicas; r++) { a += sums[(size_t)r * 2 * kFusedStatsC + c]; b += sums[(size_t)r * 2 * kFusedStatsC + kFusedStatsC + c]; }
    const double m = a / (double)F.n;
    double ss = b - m * m * (double)F.n;
    if (ss < 0) ss = 0;
    const float mean = (float)m;
    const float invstd = powf((float)(ss / (double)(F.mode == 0 ? F.n : F.n - 1)) + F.eps, -0.5f);
    if (blockIdx.x == 0) {
      if (F.mode == 0) {
        F.runningMean[c] = F.momentum * F.runningMean[c] + (1 - F.momentum) * mean;
        F.runningVar[c] = F.momentum * F.runningVar[c] + (1 - F.momentum) * (float)(ss / (double)(F.n - 1));
      }
      F.saveMean[c] = mean;
      F.saveInvStd[c] = invstd;
    }
    const float w = invstd * (F.weight ? F.weight[c] : 1.f);
    sScale[c] = w;
    sShift[c] = -mean * w + (F.bias ? F.bias[c] : 0.f);
  }
  __syncthreads();
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i0 = blockIdx.x * (long)blockDim.x + threadIdx.x; i0 < total4; i0 += 4 * stride) { // four independent 16-byte loads in flight per thread
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long i = i0 + u * stride;
      if (i < total4) v[u] = __ldg(reinterpret_cast<const float4 *>(x) + i);
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long i = i0 + u * stride;
      if (i >= total4) break;
      const int cg = (int)(i % cv);
      const float4 a = reinterpret_cast<const float4 *>(sScale)[cg], b = reinterpret_cast<const float4 *>(sShift)[cg];
      float4 o;
      o.x = fmaf(v[u].x, a.x, b.x); o.y = fmaf(v[u].y, a.y, b.y); o.z = fmaf(v[u].z, a.z, b.z); o.w = fmaf(v[u].w, a.w, b.w);
      o.x = o.x > 0 ? o.x : o.x * leak; o.y = o.y > 0 ? o.y : o.y * leak; o.z = o.z > 0 ? o.z : o.z * leak; o.w = o.w > 0 ? o.w : o.w * leak;
      if (y) reinterpret_cast<float4 *>(y)[i] = o; // y == nullptr: only the bf16 copy is consumed downstream
      if (y16) store_bf16x4(y16, i, o);
    }
  }
}
int bn_forward_from_sums(const float *x, float *y, long n, int C, const double *sums, float *saveMean, float *saveInvStd, float *runningMean,
                         float *runningVar, const float *weight, const float *bias, float eps, float momentum, int mode, float leak, cudaStream_t s, void *y16) {
  SCN_CHECK(C % 4 == 0 && C <= kFusedStatsC && (mode == 0 || mode == 2) && n > 0, "bn_forward_from_sums: unsupported configuration");
  BnFin F{n, C, mode, eps, momentum, saveMean, saveInvStd, runningMean, runningVar, weight, bias, nullptr, nullptr};
  const long total4 = n * C / 4;
  SCN_CUDA(launch_pdl(k_bn_apply_sums, dim3(stream_grid(total4, 256)), dim3(256), 0, LS(s), x, y, total4, C / 4, sums, F, leak, y16));
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// workspace: kBnReplicas x 2*kBnMaxC doubles (zero on entry, zero again on exit) + 2*kBnMaxC floats (scale, shift) + a ticket (zero)
int bn_forward(const float *x, float *y, long n, int C, float *saveMean, float *saveInvStd, float *runningMean, float *runningVar,
               const float *weight, const float *bias, float eps, float momentum, int mode, float leak, void *workspace, cudaStream_t s, void *y16) {
  double *stats = static_cast<double *>(workspace);
  float *scale = reinterpret_cast<float *>(stats + (size_t)kBnReplicas * 2 * kBnMaxC), *shift = scale + kBnMaxC; // fixed layout: the statistics area stays zero between calls
  unsigned *ticket = reinterpret_cast<unsigned *>(shift + kBnMaxC);
  BnFin F{n, C, mode, eps, momentum, saveMean, saveInvStd, runningMean, runningVar, weight, bias, scale, shift};
  SCN_CHECK(!y16 || C % 4 == 0, "bf16 shadow needs a channel count that is a multiple of 4");
  if (C % 4 == 0 && n > 0 && n <= 2048) { // small levels: statistics, finalize and apply in ONE launch
    SCN_CUDA(launch_pdl(k_bn_small, dim3(cdiv(C, 32)), dim3(256), 0, LS(s), x, y, (int)n, C, F, leak, y16));
    SCN_CUDA(cudaGetLastError());
    return 0;
  }
  bool finalized = false;
  if (mode != 1 && n > 0) {
    // every CTA ends with one double atomic per channel, and atomics to one address serialise (~45 ns each, measured:
    // 1073 CTAs -> 48 us for a 17 MB input): at most 4 CTAs per SM, >= 256 rows each, spread over kBnReplicas accumulators
    int rowsPerCta = (int)std::max<long>(256, (n + kSMs * 4 - 1) / (kSMs * 4));
    int grid = cdiv(n, rowsPerCta);
    double *part = nullptr; // deterministic mode: per-CTA sums, added in CTA order into replica 0 (k_bn_finalize reads it)
    if (deterministic()) SCN_TRY(det_scratch(s, (size_t)grid * 2 * C * sizeof(double), (void **)&part));
    else ++g_counters[kCntFloatAtomic];
    if (C % 4 == 0) {
      SCN_CHECK(C / 4 <= 256, "BatchNorm: more than 1024 channels not supported");
      k_bn_stats<<<grid, 256, 2 * 256 * 16, LS(s)>>>(x, n, C, rowsPerCta, stats, ticket, F, part); // last CTA finalizes
      finalized = !part;
    } else {
      SCN_CHECK(C <= 256, "BatchNorm: channel count not a multiple of 4 must be <= 256");
      k_bn_stats_scalar<<<grid, 256, 0, LS(s)>>>(x, n, C, rowsPerCta, stats, part);
    }
    if (part) SCN_TRY(ordered_sum(part, grid, 2l * C, stats, s));
  }
  if (!finalized) k_bn_finalize<<<cdiv(C, 128), 128, 0, LS(s)>>>(stats, F);
  if (n) {
    long total = n * C;
    if (C % 4 == 0) k_bn_apply<<<stream_grid(total / 4, 256), 256, 0, LS(s)>>>(x, y, total / 4, C / 4, scale, shift, leak, y16);
    else k_bn_apply_scalar<<<stream_grid(total, 256), 256, 0, LS(s)>>>(x, y, total, C, scale, shift, leak);
  }
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ BN backward
// BatchNormalization_BackwardPass (SCN/CPU/BatchNormalization.cpp:64-107).  Pass 1: d = dy * (y>0?1:leak)
// written back into dy (the reference rewrites d_output in place, :79-82), per-channel sum d and
// sum (x-mean)*d.  Pass 2: dx = (d - mean(d) - (x-mean)*k) * invstd * gamma.
__global__ void __launch_bounds__(256) k_bn_bwd_stats(const float *__restrict__ x, const float *__restrict__ y, float *__restrict__ dy, long n, int C,
                                                      int rowsPerCta, const float *__restrict__ saveMean, float leak, double *__restrict__ stats,
                                                      double *__restrict__ part) {
  __shared__ float S[256], Q[256];
  const int tid = threadIdx.x;
  const int cols = min(C, 256), rowLanes = 256 / cols;
  const long r0 = (long)blockIdx.x * rowsPerCta, r1 = min(n, r0 + rowsPerCta);
  for (int cb = 0; cb < C; cb += cols) {
    const int c = cb + tid % cols, rl = tid / cols;
    float s = 0.f, q = 0.f;
    if (rl < rowLanes && c < C) {
      const float m = saveMean[c];
      for (long r = r0 + rl; r < r1; r += rowLanes) {
        long i = r * C + c;
        float d = dy[i] * (y[i] > 0 ? 1.f : leak);
        dy[i] = d;
        s += d;
        q = fmaf(x[i] - m, d, q);
      }
    }
    S[tid] = s; Q[tid] = q;
    __syncthreads();
    if (tid < cols && cb + tid < C) {
      double a = 0, b = 0;
      for (int l = 0; l < rowLanes; l++) { a += S[l * cols + tid]; b += Q[l * cols + tid]; }
      if (part) { part[(size_t)blockIdx.x * 2 * C + cb + tid] = a; part[(size_t)blockIdx.x * 2 * C + C + cb + tid] = b; }
      else { atomicAdd(stats + cb + tid, a); atomicAdd(stats + C + cb + tid, b); }
    }
    __syncthreads();
  }
}
__global__ void k_bn_bwd_finalize(const double *__restrict__ stats, long n, int C, const float *__restrict__ saveInvStd, float *dWeight, float *dBias,
                                  float *gradMean, float *kk) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float gm = (float)stats[c], dotp = (float)stats[C + c];
  if (dBias) dBias[c] = gm;
  if (dWeight) dWeight[c] = dotp * saveInvStd[c];
  gradMean[c] = gm / (float)n;
  kk[c] = dotp * saveInvStd[c] * saveInvStd[c] / (float)n;
}
__global__ void __launch_bounds__(256) k_bn_bwd_apply(const float *__restrict__ x, const float *__restrict__ d, float *__restrict__ dx, long total, int C,
                                                      const float *__restrict__ saveMean, const float *__restrict__ saveInvStd,
                                                      const float *__restrict__ weight, const float *__restrict__ gradMean, const float *__restrict__ kk) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    dx[i] = (d[i] - gradMean[c] - (x[i] - saveMean[c]) * kk[c]) * saveInvStd[c] * (weight ? weight[c] : 1.f);
  }
}
// float4 versions (C % 4 == 0): four channels per thread, two rows in flight -- the scalar kernels above ran at well under half of
// the HBM rate (one 4-byte access in flight per thread, an integer modulo per element in the apply pass).
// y16 (optional): the BatchNorm output as bf16 rows -- only its sign is needed (the leaky-ReLU mask), and a replayed training step in
// bf16 mode never writes the fp32 output rows of a BatchNorm whose only readers are tensor-core convolutions.
__device__ __forceinline__ float4 bn_y4(const float4 *y, const uint2 *y16, long i) {
  if (!y16) return y[i];
  const uint2 v = y16[i]; // bf16 = the upper half of the fp32 pattern: the sign survives a plain shift
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xffff0000u));
}
__global__ void __launch_bounds__(256) k_bn_bwd_stats4(const float4 *__restrict__ x, const float4 *__restrict__ y, const uint2 *__restrict__ y16, float4 *__restrict__ dy, long n, int C4,
                                                       int rowsPerCta, const float *__restrict__ saveMean, float leak, double *__restrict__ stats,
                                                       double *__restrict__ part) {
  __shared__ float4 S[256], Q[256];
  const int tid = threadIdx.x;
  const int cols = min(C4, 256), rowLanes = 256 / cols;
  const long r0 = (long)blockIdx.x * rowsPerCta, r1 = min(n, r0 + rowsPerCta);
  for (int cb = 0; cb < C4; cb += cols) {
    const int c = cb + tid % cols, rl = tid / cols;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
    if (rl < rowLanes && c < C4) {
      const float4 m = __ldg(reinterpret_cast<const float4 *>(saveMean) + c);
      auto one = [&](const float4 &xv, const float4 &yv, float4 d) {
        d.x *= yv.x > 0 ? 1.f : leak; d.y *= yv.y > 0 ? 1.f : leak; d.z *= yv.z > 0 ? 1.f : leak; d.w *= yv.w > 0 ? 1.f : leak;
        s.x += d.x; s.y += d.y; s.z += d.z; s.w += d.w;
        q.x = fmaf(xv.x - m.x, d.x, q.x); q.y = fmaf(xv.y - m.y, d.y, q.y); q.z = fmaf(xv.z - m.z, d.z, q.z); q.w = fmaf(xv.w - m.w, d.w, q.w);
        return d;
      };
      long r = r0 + rl;
      for (; r + rowLanes < r1; r += 2 * rowLanes) { // two rows in flight
        const long i0 = r * C4 + c, i1 = (r + rowLanes) * C4 + c;
        const float4 x0 = x[i0], y0 = bn_y4(y, y16, i0), d0 = dy[i0], x1 = x[i1], y1 = bn_y4(y, y16, i1), d1 = dy[i1];
        dy[i0] = one(x0, y0, d0);
        dy[i1] = one(x1, y1, d1);
      }
      if (r < r1) { const long i0 = r * C4 + c; dy[i0] = one(x[i0], bn_y4(y, y16, i0), dy[i0]); }
    }
    S[tid] = s; Q[tid] = q;
    __syncthreads();
    if (tid < cols && cb + tid < C4) {
      double a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
      for (int l = 0; l < rowLanes; l++) {
        const float4 sv = S[l * cols + tid], qv = Q[l * cols + tid];
        a[0] += sv.x; a[1] += sv.y; a[2] += sv.z; a[3] += sv.w;
        b[0] += qv.x; b[1] += qv.y; b[2] += qv.z; b[3] += qv.w;
      }
      const int ch = (cb + tid) * 4, C = C4 * 4;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (part) { part[(size_t)blockIdx.x * 2 * C + ch + j] = a[j]; part[(size_t)blockIdx.x * 2 * C + C + ch + j] = b[j]; }
        else { atomicAdd(stats + ch + j, a[j]); atomicAdd(stats + C + ch + j, b[j]); }
      }
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) k_bn_bwd_apply4(const float4 *__restrict__ x, const float4 *__restrict__ d, float4 *__restrict__ dx, long total4, int C4,
                                                       const float *__restrict__ saveMean, const float *__restrict__ saveInvStd,
                                                       const float *__restrict__ weight, const float *__restrict__ gradMean, const float *__restrict__ kk) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total4; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4);
    const float4 m = __ldg(reinterpret_cast<const float4 *>(saveMean) + c), is = __ldg(reinterpret_cast<const float4 *>(saveInvStd) + c);
    const float4 gm = __ldg(reinterpret_cast<const float4 *>(gradMean) + c), k4 = __ldg(reinterpret_cast<const float4 *>(kk) + c);
    const float4 w = weight ? __ldg(reinterpret_cast<const float4 *>(weight) + c) : make_float4(1.f, 1.f, 1.f, 1.f);
    const float4 xv = x[i], dv = d[i];
    float4 o;
    o.x = (dv.x - gm.x - (xv.x - m.x) * k4.x) * is.x * w.x;
    o.y = (dv.y - gm.y - (xv.y - m.y) * k4.y) * is.y * w.y;
    o.z = (dv.z - gm.z - (xv.z - m.z) * k4.z) * is.z * w.z;
    o.w = (dv.w - gm.w - (xv.w - m.w) * k4.w) * is.w * w.w;
    dx[i] = o;
  }
}
int bn_backward(const float *x, float *dx, const float *y, float *dy, long n, int C, const float *saveMean, const float *saveInvStd,
                const float *weight, float *dWeight, float *dBias, float leak, void *workspace, cudaStream_t s, const void *y16) {
  double *stats = static_cast<double *>(workspace);
  float *gradMean = reinterpret_cast<float *>(stats + 2 * C), *kk = gradMean + C;
  SCN_CUDA(cudaMemsetAsync(stats, 0, 2 * C * sizeof(double), s));
  SCN_CHECK(y || y16, "BatchNorm backward needs the output rows (fp32 or bf16)");
  const bool vec = C % 4 == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(y16) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx) |
                                  reinterpret_cast<uintptr_t>(saveMean) | reinterpret_cast<uintptr_t>(saveInvStd) | reinterpret_cast<uintptr_t>(weight)) & 15) == 0;
  if (n) {
    int rowsPerCta = (int)std::max<long>(64, (n + kSMs * 16 - 1) / (kSMs * 16));
    const int grid = cdiv(n, rowsPerCta);
    SCN_CHECK(vec || y, "BatchNorm backward: the bf16-only output path needs 16-byte aligned rows of a multiple of 4 channels");
    double *part = nullptr; // deterministic mode: per-CTA sums, added in CTA order
    if (deterministic()) SCN_TRY(det_scratch(s, (size_t)grid * 2 * C * sizeof(double), (void **)&part));
    else ++g_counters[kCntFloatAtomic];
    if (vec) k_bn_bwd_stats4<<<grid, 256, 0, LS(s)>>>(reinterpret_cast<const float4 *>(x), reinterpret_cast<const float4 *>(y), y ? nullptr : static_cast<const uint2 *>(y16),
                                                      reinterpret_cast<float4 *>(dy), n, C / 4, rowsPerCta, saveMean, leak, stats, part);
    else k_bn_bwd_stats<<<grid, 256, 0, LS(s)>>>(x, y, dy, n, C, rowsPerCta, saveMean, leak, stats, part);
    if (part) SCN_TRY(ordered_sum(part, grid, 2l * C, stats, s));
  }
  k_bn_bwd_finalize<<<cdiv(C, 128), 128, 0, LS(s)>>>(stats, n, C, saveInvStd, dWeight, dBias, gradMean, kk);
  if (n && vec) k_bn_bwd_apply4<<<stream_grid(n * C / 4, 256), 256, 0, LS(s)>>>(reinterpret_cast<const float4 *>(x), reinterpret_cast<const float4 *>(dy), reinterpret_cast<float4 *>(dx),
                                                                                n * C / 4, C / 4, saveMean, saveInvStd, weight, gradMean, kk);
  else if (n) k_bn_bwd_apply<<<stream_grid(n * C, 256), 256, 0, LS(s)>>>(x, dy, dx, n * C, C, saveMean, saveInvStd, weight, gradMean, kk);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ InputLayer
// InputLayer_ForwardPass (SCN/CPU/IOLayers.cpp:11-29): out[row] = sum_i mult * in[rules[row][i]], rows in list order.
__global__ void __launch_bounds__(256) k_input_fwd(const float *__restrict__ in, float *__restrict__ out, int nOut, int w, int C, const int *__restrict__ tab, int average) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < (long)nOut * C; i += (long)gridDim.x * blockDim.x) {
    int row = (int)(i / C), c = (int)(i % C);
    const int *r = tab + (long)row * w;
    int na = r[0];
    float mult = (average && na > 0) ? 1.f / na : 1.f;
    float acc = 0.f;
    for (int j = 1; j <= na; j++) acc += mult * __ldg(in + (long)r[j] * C + c);
    out[i] = acc;
  }
}
// mode 0: rows are unique; out row id <- first-occurrence order == input order
__global__ void __launch_bounds__(256) k_input_bwd(float *__restrict__ din, const float *__restrict__ dout, int nOut, int w, int C, const int *__restrict__ tab, int average) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < (long)nOut * C; i += (long)gridDim.x * blockDim.x) {
    int row = (int)(i / C), c = (int)(i % C);
    const int *r = tab + (long)row * w;
    int na = r[0];
    float mult = (average && na > 0) ? 1.f / na : 1.f;
    float g = mult * dout[i];
    for (int j = 1; j <= na; j++) din[(long)r[j] * C + c] = g; // an input row feeds exactly one voxel: plain store
  }
}
// Same, plus a bf16 copy of the output rows zero-padded to Cp channels (the packed operand of the first convolution in
// bf16 mode, which otherwise needs a separate padding pass over the rows).
// One thread per output row: the rule-table entries are read once per row (not once per channel) and the bf16 row
// (Cp <= 32 channels) leaves as 16-byte stores.
__global__ void __launch_bounds__(256) k_input_fwd_pad16(const float *__restrict__ in, float *__restrict__ out, __nv_bfloat16 *__restrict__ out16, int nOut, int w,
                                                         int C, int Cp, const int *__restrict__ tab, int average) {
  for (long row = blockIdx.x * (long)blockDim.x + threadIdx.x; row < nOut; row += (long)gridDim.x * blockDim.x) {
    const int *r = tab + row * w;
    const int na = r[0];
    const float mult = (average && na > 0) ? 1.f / na : 1.f;
    float acc[32];
#pragma unroll
    for (int c = 0; c < 32; c++) acc[c] = 0.f;
    for (int j = 1; j <= na; j++) {
      const float *src = in + (long)r[j] * C;
#pragma unroll
      for (int c = 0; c < 32; c++)
        if (c < C) acc[c] += mult * __ldg(src + c);
    }
#pragma unroll
    for (int c = 0; c < 32; c++)
      if (c < C) out[row * C + c] = acc[c];
    uint4 *dst = reinterpret_cast<uint4 *>(out16 + row * Cp);
#pragma unroll
    for (int q = 0; q < 4; q++) {
      if (q * 8 >= Cp) break;
      __nv_bfloat162 v0 = __floats2bfloat162_rn(acc[q * 8], acc[q * 8 + 1]), v1 = __floats2bfloat162_rn(acc[q * 8 + 2], acc[q * 8 + 3]);
      __nv_bfloat162 v2 = __floats2bfloat162_rn(acc[q * 8 + 4], acc[q * 8 + 5]), v3 = __floats2bfloat162_rn(acc[q * 8 + 6], acc[q * 8 + 7]);
      uint4 pk;
      pk.x = *reinterpret_cast<unsigned int *>(&v0); pk.y = *reinterpret_cast<unsigned int *>(&v1);
      pk.z = *reinterpret_cast<unsigned int *>(&v2); pk.w = *reinterpret_cast<unsigned int *>(&v3);
      dst[q] = pk;
    }
  }
}
int input_forward_pad16(const float *in, float *out, void *out16, int nOut, int maxActive, int C, int Cp, const int *tab, int average, cudaStream_t s) {
  SCN_CHECK(C <= 32 && Cp <= 32 && Cp % 8 == 0 && Cp >= C, "input_forward_pad16: at most 32 channels");
  if (nOut) k_input_fwd_pad16<<<stream_grid(nOut, 256, 16), 256, 0, LS(s)>>>(in, out, static_cast<__nv_bfloat16 *>(out16), nOut, 1 + maxActive, C, Cp, tab, average);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
int input_forward(const float *in, float *out, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s) {
  if (nOut) k_input_fwd<<<stream_grid((long)nOut * C, 256), 256, 0, LS(s)>>>(in, out, nOut, 1 + maxActive, C, tab, average);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
int input_backward(float *din, const float *dout, long nIn, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s) {
  SCN_CUDA(cudaMemsetAsync(din, 0, nIn * C * sizeof(float), s)); // rows dropped by modes 1/2 get zero gradient
  if (nOut) k_input_bwd<<<stream_grid((long)nOut * C, 256), 256, 0, LS(s)>>>(din, dout, nOut, 1 + maxActive, C, tab, average);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ add_feature_planes / AddTable
__global__ void __launch_bounds__(256) k_add(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ o, long n, void *__restrict__ o16) {
  long n4 = n >> 2;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 u = __ldg(reinterpret_cast<const float4 *>(a) + i), v = __ldg(reinterpret_cast<const float4 *>(b) + i);
    float4 r = make_float4(u.x + v.x, u.y + v.y, u.z + v.z, u.w + v.w);
    reinterpret_cast<float4 *>(o)[i] = r;
    if (o16) store_bf16x4(o16, i, r);
  }
  for (long i = (n4 << 2) + blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) o[i] = a[i] + b[i];
}
int add_rows(const float *a, const float *b, float *o, long n, cudaStream_t s, void *o16) {
  SCN_CHECK(!o16 || n % 4 == 0, "bf16 shadow needs an element count that is a multiple of 4");
  if (n) k_add<<<stream_grid(n / 4 + 1, 256), 256, 0, LS(s)>>>(a, b, o, n, o16);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

} // namespace scn
