// What the translation units of the library call in each other: convolution launchers, row operations, internal entries (capi.cu).
#pragma once
#include "common.cuh"

struct scn_metadata;

namespace scn {

// A lateral 1x1x1 convolution folded into a convolution, out = conv(x) [+ addend] + in[row] @ w (scn_fuse_next_lateral); in == nullptr: none
struct Lateral { const float *in; const void *in16; const float *w; long long tag; int Cin; long rows; };
// What a forward convolution is asked to fold into its tensor-core launch; a launch that cannot take a part ignores it.
struct ConvFusion {
  Lateral lat = {nullptr, nullptr, nullptr, 0, 0, 0};
  double *stats = nullptr;     // [kBnReplicas][2][kFusedStatsC], zeroed by the caller: per-channel sum / sum of squares of the output
  const void *pad16 = nullptr; // 16-bit copy of the input rows already zero-padded to padC channels (written by the input layer)
  int padC = 0;
};
// Which parts of a ConvFusion a call took.
struct ConvFused { bool lateral = false, stats = false; };

// ---------------------------------------------------------------- tensor-core convolution (conv_tc.cu)
// One launch of the output-stationary tensor-core convolution over an execution plan.
struct TcConv {
  const float *in = nullptr;  // fp32 input rows; in16 (optional): their 16-bit copy in the mode's format, used when Cin is a multiple of 64
  const void *in16 = nullptr;
  long nInRows = 0;
  const float *W = nullptr;   // [nWeights][CinW][Cout], or transposed (wT = 1: [K][Cout][CinW]; wT = 2: offsets reversed as well)
  long long wTag = 0;         // content tag of W for the weight-image cache (0: not cached)
  int nWeights = 0, CinW = 0, wT = 0; // CinW = 0: Cin
  const int *nbr = nullptr, *outRow = nullptr;
  const unsigned long long *tileMask = nullptr;
  const int *tileW = nullptr; // deconvolution plans: weight slice per tile (then K == 1)
  int nOut = 0, K = 0;        // plan sites and filter offsets
  int Cin = 0, Cout = 0;
  const float *bias = nullptr, *addend = nullptr; // addend (optional, [output rows][Cout]): out = conv + addend
  float *out = nullptr;
  void *out16 = nullptr;      // optional: the result in the mode's 16-bit format
  long nOutRows = 0;
  int mathMode = 0;           // scn_set_math_mode: 1 = TF32, 2 = BF16, 3 = TF32X3, 5 = F16 operands (narrow layers keep TF32 in modes 2 and 5)
  // column slab of a layer wider than 256 output channels (launch_conv_plan_tc_slabs): this launch computes output columns
  // [col0, col0 + Cout) of rows ldOut wide -- out, addend, out16 and bias are full-width, W is [..][ldOut] (0: Cout, no slab)
  int col0 = 0, ldOut = 0;
  ConvFusion fuse;
  ConvFused *fused = nullptr; // optional: set where the launch took a part of `fuse`
};
int launch_conv_plan_tc(const TcConv &c, cudaStream_t s);
int launch_conv_dw_tc(const float *in, const float *d_out, float *dW, const int2 *pairs, const int *d_off, const int *offHost, int K, long nInRows,
                      long nOutRows, int Cin, int Cout, int srcIsY, int mathMode, cudaStream_t s, const void *in16, const void *dout16,
                      const int *planNbr, const int *planOutRow, const unsigned long long *planMask, int planPos);
int tc_available();
bool dw_tc_ok(int Cin, int Cout, int K, int mathMode);
bool dw_plan_ok(int Cin, int Cout, int K, int mathMode);
int to_16(const float *x, void *y, long n, cudaStream_t s);
int from_16(const void *x, float *y, long n, cudaStream_t s);
int dout16_copy(const float *d_out, long n, cudaStream_t s, const void **out);
long release_conv_caches();

// ---------------------------------------------------------------- CUDA-core convolution (conv_simt.cu, conv_bwd.cu)
int launch_conv_plan_simt(const float *in, float *out, const float *W, const int *nbr, const int *outRow, int nOut, int K, int Cin, int Cout,
                          const float *bias, cudaStream_t s);
int launch_conv_list_simt(const float *in, float *out, const float *W, const int2 *pairs, const int *d_off, const int *offHost, int K, int Cin,
                          int Cout, int srcIsY, int singlePass, cudaStream_t s);
int conv_backward_simt(const float *in, float *d_in, const float *d_out, const float *W, float *dW, float *d_bias, const int2 *pairs,
                       const int *d_off, const int *offHost, int K, long nInRows, long nOutRows, int Cin, int Cout, int srcIsY, cudaStream_t s, int skipDIn,
                       int mathMode, const void *in16, const void *dout16, const int *planNbr, const int *planOutRow, const unsigned long long *planMask,
                       int planPos);
int transpose_weights(const float *W, float *Wt, int K, int Cin, int Cout, int reverse, cudaStream_t s);
int dense_rows_dw(const float *in, const float *d_out, float *dW, float *d_bias, long n, int Cin, int Cout, cudaStream_t s);

// ---------------------------------------------------------------- row operations (rowops.cu)
int bn_forward(const float *x, float *y, long n, int C, float *saveMean, float *saveInvStd, float *runningMean, float *runningVar,
               const float *weight, const float *bias, float eps, float momentum, int mode, float leak, void *workspace, cudaStream_t s, void *y16);
int bn_forward_from_sums(const float *x, float *y, long n, int C, const double *sums, float *saveMean, float *saveInvStd, float *runningMean,
                         float *runningVar, const float *weight, const float *bias, float eps, float momentum, int mode, float leak, cudaStream_t s, void *y16);
int bn_backward(const float *x, float *dx, const float *y, float *dy, long n, int C, const float *saveMean, const float *saveInvStd,
                const float *weight, float *dWeight, float *dBias, float leak, void *workspace, cudaStream_t s, const void *y16);
int input_forward(const float *in, float *out, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s);
int input_forward_pad16(const float *in, float *out, void *out16, int nOut, int maxActive, int C, int Cp, const int *tab, int average, cudaStream_t s);
int input_backward(float *din, const float *dout, long nIn, int nOut, int maxActive, int C, const int *tab, int average, cudaStream_t s);
int add_rows(const float *a, const float *b, float *o, long n, cudaStream_t s, void *o16);

// ---------------------------------------------------------------- internal entries (capi.cu)
// The scn_*_convolution_forward entries with an explicit fusion request; `fused` (optional) reports what was taken.
int submanifold_forward(scn_metadata *m, const long sz[3], const long f[3], const float *in, float *out, const float *w, const float *bias, int Cin,
                        int Cout, double *macs, const void *in_bf16, long long weight_tag, const float *add_in, void *out_bf16, const ConvFusion &fuse,
                        ConvFused *fused);
int convolution_forward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in, float *out,
                        const float *w, const float *bias, int Cin, int Cout, double *macs, const void *in_bf16, long long weight_tag, const float *add_in,
                        void *out_bf16, const ConvFusion &fuse, ConvFused *fused);
int deconvolution_forward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in, float *out,
                          const float *w, const float *bias, int Cin, int Cout, double *macs, const void *in_bf16, long long weight_tag, const float *add_in,
                          void *out_bf16, const ConvFusion &fuse, ConvFused *fused);
// The scn_*_convolution_backward entries with the forward's 16-bit copy of `in` (whole rows, the mode's format; may be null), from
// which the weight-gradient kernel gathers instead of converting the fp32 rows again.
int submanifold_backward(scn_metadata *m, const long sz[3], const long f[3], const float *in, float *d_in, const float *d_out, const float *w,
                         float *dw, float *d_bias, int Cin, int Cout, const void *in16);
int convolution_backward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in, float *d_in,
                         const float *d_out, const float *w, float *dw, float *d_bias, int Cin, int Cout, const void *in16);
int deconvolution_backward(scn_metadata *m, const long inS[3], const long outS[3], const long f[3], const long st[3], const float *in, float *d_in,
                           const float *d_out, const float *w, float *dw, float *d_bias, int Cin, int Cout, const void *in16);
bool backward_reads_lists(int kind, const long *f, const long *st, int Cin, int Cout, bool wantDIn);
int batchnorm_backward_y16(const float *in, float *d_in, const float *out, const void *out_bf16, float *d_out, long n, int C, const float *save_mean,
                           const float *save_invstd, const float *weight, float *d_weight, float *d_bias, float leak, cudaStream_t s);
int build_subm_on_caller(scn_metadata *m, const long *sz, const long *f);
cudaStream_t metadata_stream(scn_metadata *m);

} // namespace scn
