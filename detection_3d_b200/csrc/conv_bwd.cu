// Backward of the three convolution kinds (fp32 CUDA cores).
//   dIn  = sum_k scatter( gather(dOut, rules_k.dst) @ W[k]^T )   -> in tf32 / bf16 mode the tcgen05 FORWARD kernel on
//          (dOut, W^T): the submanifold plan is symmetric (dIn[q] = sum_j dOut[nbr[q][j]] @ W[K-1-j]^T), the input
//          gradient of a strided convolution is a deconvolution and vice versa (capi.cu); in fp32 mode the forward list kernel run on
//          (dOut, W^T) with the pair columns swapped, lists back to back (a source row occurs at
//          most once per list, so the read-modify-write is race free, as in the reference).
//   dW[k] = gather(in, rules_k.src)^T @ gather(dOut, rules_k.dst) -> split over rule chunks, fp32
//          atomics into dW (replaces dConvolution_KMxKN_backward_dW_A/B, SCN/CUDA/Convolution.cu:249-410); in deterministic mode
//          each chunk stores its partial dW[k] into its own slot and ordered_sum adds the chunks in chunk order.
// Reference semantics: SCN/CPU/Convolution.cpp:81-115,152-185, SCN/CPU/Deconvolution.cpp:43-77.
#include "common.cuh"

namespace scn {
int launch_conv_list_simt(const float *in, float *out, const float *W, const int2 *pairs, const int *d_off, const int *offHost, int K, int Cin,
                          int Cout, int srcIsY, int singlePass, cudaStream_t s);
int launch_conv_dw_tc(const float *in, const float *d_out, float *dW, const int2 *pairs, const int *d_off, const int *offHost, int K, long nInRows,
                      long nOutRows, int Cin, int Cout, int srcIsY, int mathMode, cudaStream_t s, const void *in16, const void *dout16,
                      const int *planNbr, const int *planOutRow, const unsigned long long *planMask, int planPos);

// Wt[k'][co][ci] = W[k][ci][co], k' = k or (reverse) K - 1 - k
__global__ void k_transpose_w(const float *__restrict__ W, float *__restrict__ Wt, int K, int Cin, int Cout, int reverse) {
  long n = (long)K * Cin * Cout;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int co = (int)(i % Cout);
    long t = i / Cout;
    int ci = (int)(t % Cin), k = (int)(t / Cin);
    Wt[((long)(reverse ? K - 1 - k : k) * Cout + co) * Cin + ci] = W[i];
  }
}
int transpose_weights(const float *W, float *Wt, int K, int Cin, int Cout, int reverse, cudaStream_t s) {
  k_transpose_w<<<stream_grid((long)K * Cin * Cout, 256), 256, 0, LS(s)>>>(W, Wt, K, Cin, Cout, reverse);
  SCN_CUDA(cudaGetLastError());
  return 0;
}

constexpr int BM = 64, BN = 64, BK = 16, BPAD = 4;
__global__ void __launch_bounds__(256) k_dw(const float *__restrict__ in, const float *__restrict__ dOut, float *__restrict__ dW, const int2 *__restrict__ pairs,
                                            int start, int len, int chunk, int Cin, int Cout, int srcIsY, float *__restrict__ part) {
  __shared__ __align__(16) float A_s[BK][BM + BPAD];
  __shared__ __align__(16) float B_s[BK][BN];
  __shared__ int s_src[BK], s_dst[BK];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int ci0 = blockIdx.y * BM, co0 = blockIdx.z * BN;
  const int i0 = blockIdx.x * chunk, i1 = min(len, i0 + chunk);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;
  for (int ib = i0; ib < i1; ib += BK) {
    __syncthreads();
    if (tid < BK) {
      int2 pr = make_int2(-1, -1);
      if (ib + tid < i1) pr = pairs ? __ldg(pairs + start + ib + tid) : make_int2(start + ib + tid, start + ib + tid); // no list: dense rows
      s_src[tid] = srcIsY ? pr.y : pr.x;
      s_dst[tid] = srcIsY ? pr.x : pr.y;
    }
    __syncthreads();
    // 16 rules x 64 channels each side: 1024 floats, 4 per thread
    {
      const int kk = tid >> 4, c4 = (tid & 15) * 4;
      const int sr = s_src[kk], dr = s_dst[kk];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        int ci = ci0 + c4 + j, co = co0 + c4 + j;
        A_s[kk][c4 + j] = (sr >= 0 && ci < Cin) ? __ldg(in + (long)sr * Cin + ci) : 0.f;
        B_s[kk][c4 + j] = (dr >= 0 && co < Cout) ? __ldg(dOut + (long)dr * Cout + co) : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; kk++) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; i++) a[i] = A_s[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; j++) b[j] = B_s[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      int ci = ci0 + ty * 4 + i, co = co0 + tx * 4 + j;
      if (ci < Cin && co < Cout) {
        if (part) part[((long)blockIdx.x * Cin + ci) * Cout + co] = acc[i][j];
        else atomicAdd(dW + (long)ci * Cout + co, acc[i][j]);
      }
    }
}
__global__ void k_colsum(const float *__restrict__ x, long n, int C, float *__restrict__ out, float *__restrict__ part) {
  int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (long r = blockIdx.x; r < n; r += gridDim.x) s += x[r * C + c];
  if (part) part[(long)blockIdx.x * C + c] = s;
  else atomicAdd(out + c, s);
}
// d_bias = column sums of d_out (zeroed by the caller)
static int column_sums(const float *d_out, long n, int C, float *d_bias, cudaStream_t s) {
  if (!n) return 0;
  const int parts = kSMs * 2;
  float *part = nullptr;
  if (deterministic()) SCN_TRY(det_scratch(s, (size_t)parts * C * 4, (void **)&part));
  else ++g_counters[kCntFloatAtomic];
  k_colsum<<<dim3(parts, cdiv(C, 128)), 128, 0, LS(s)>>>(d_out, n, C, d_bias, part);
  if (part) SCN_TRY(ordered_sum(part, parts, (long)C, d_bias, s));
  SCN_CUDA(cudaGetLastError());
  return 0;
}
// dW (zeroed by the caller) += the chunks of one rule list (pairs == nullptr: dense rows, row i pairs with row i)
static int dw_chunks(const float *in, const float *d_out, float *dW, const int2 *pairs, int start, int len, int Cin, int Cout, int srcIsY, cudaStream_t s) {
  int chunk = std::max(256, cdiv(len, kSMs * 4));
  chunk = (chunk + BK - 1) / BK * BK;
  dim3 grid(cdiv(len, chunk), cdiv(Cin, BM), cdiv(Cout, BN));
  float *part = nullptr;
  if (deterministic()) SCN_TRY(det_scratch(s, (size_t)grid.x * Cin * Cout * 4, (void **)&part));
  else ++g_counters[kCntFloatAtomic];
  k_dw<<<grid, 256, 0, LS(s)>>>(in, d_out, dW, pairs, start, len, chunk, Cin, Cout, srcIsY, part);
  if (part) SCN_TRY(ordered_sum(part, (int)grid.x, (long)Cin * Cout, dW, s));
  SCN_CUDA(cudaGetLastError());
  return 0;
}

// NetworkInNetwork_accGradParameters (SCN/CPU/NetworkInNetwork.cpp:36-46): dW = in^T @ d_out over dense rows (row i pairs with row i),
// d_bias = column sums of d_out.  Both overwritten.
int dense_rows_dw(const float *in, const float *d_out, float *dW, float *d_bias, long n, int Cin, int Cout, cudaStream_t s) {
  SCN_CUDA(cudaMemsetAsync(dW, 0, (size_t)Cin * Cout * 4, s));
  if (d_bias) {
    SCN_CUDA(cudaMemsetAsync(d_bias, 0, (size_t)Cout * 4, s));
    SCN_TRY(column_sums(d_out, n, Cout, d_bias, s));
  }
  if (n == 0) return 0;
  return dw_chunks(in, d_out, dW, nullptr, 0, (int)n, Cin, Cout, 0, s);
}

// skipDIn: the caller computes d_in itself (tensor-core forward kernel on (d_out, W^T)); only dW / d_bias here
int conv_backward_simt(const float *in, float *d_in, const float *d_out, const float *W, float *dW, float *d_bias, const int2 *pairs,
                       const int *d_off, const int *offHost, int K, long nInRows, long nOutRows, int Cin, int Cout, int srcIsY, cudaStream_t s, int skipDIn, int mathMode,
                       const void *in16, const void *dout16, const int *planNbr, const int *planOutRow, const unsigned long long *planMask, int planPos) {
  if (!skipDIn) SCN_CUDA(cudaMemsetAsync(d_in, 0, (size_t)nInRows * Cin * 4, s));
  SCN_CUDA(cudaMemsetAsync(dW, 0, (size_t)K * Cin * Cout * 4, s));
  if (d_bias) {
    SCN_CUDA(cudaMemsetAsync(d_bias, 0, (size_t)Cout * 4, s));
    SCN_TRY(column_sums(d_out, nOutRows, Cout, d_bias, s));
  }
  // pairs == nullptr: the caller did not build the rule lists (input gradient done / not wanted, weight gradient from the plan)
  if (pairs && offHost[K] == 0) return 0;
  if (!pairs && (!skipDIn || !planNbr || mathMode == 0)) { set_error("convolution backward: rule lists missing"); return -2; }
  if (!skipDIn) {
    float *Wt = nullptr;
    SCN_CUDA(cudaMallocAsync((void **)&Wt, (size_t)K * Cin * Cout * 4, s));
    k_transpose_w<<<stream_grid((long)K * Cin * Cout, 256), 256, 0, LS(s)>>>(W, Wt, K, Cin, Cout, 0);
    // dIn: rows of d_out gathered by the forward destination column, scattered to the forward source column
    int r = launch_conv_list_simt(d_out, d_in, Wt, pairs, d_off, offHost, K, Cout, Cin, !srcIsY, /*singlePass=*/0, s);
    cudaFreeAsync(Wt, s);
    if (r) return r;
  }
  if (mathMode != 0) { // weight gradient on the tensor cores where the channel counts allow (conv_tc.cu, conv_dw_tc)
    int r = launch_conv_dw_tc(in, d_out, dW, pairs, d_off, offHost, K, nInRows, nOutRows, Cin, Cout, srcIsY, mathMode, s, in16, dout16, planNbr, planOutRow, planMask, planPos);
    if (r <= 0) return r;
  }
  if (!pairs) { set_error("convolution backward: rule lists missing for the CUDA-core weight gradient"); return -2; }
  for (int L_ = 0; L_ < K; L_++) {
    int len = offHost[L_ + 1] - offHost[L_];
    if (!len) continue;
    SCN_TRY(dw_chunks(in, d_out, dW + (long)L_ * Cin * Cout, pairs, offHost[L_], len, Cin, Cout, srcIsY, s));
  }
  SCN_CUDA(cudaGetLastError());
  return 0;
}
} // namespace scn
