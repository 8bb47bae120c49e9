// SparseToDense: the active rows of one spatial size scattered into a zero-filled dense tensor [batch][planes][X][Y][Z].
//   reference: sparseconvnet/sparseToDense.py:25-78 (module), SCN/CPU/SparseToDense.cpp:7-101, SCN/CUDA/SparseToDense.cu:9-69,
//   rules SCN/Metadata/ConvolutionRules.h:109-151 (one (row, spatial offset) pair per active site, hash-iteration order -- the order
//   does not affect the result), caller layers/roi_align_rotated_3d.py:81 and sparseconvnet/tools_3d_2d.py:7-48.
// HBM bound by the dense output: planes x volume x 4 bytes are zero-filled whatever the occupancy, the scatter itself moves
// 2 x 4 x n x planes bytes.  32 sites (in spatial order: neighbours along z are adjacent cells) x 32 planes go through a shared-
// memory transpose, so the row reads (plane-contiguous) and the dense writes (cell-contiguous) are both coalesced.
#include "../../include/scn_b200.h"
#include "metadata.cuh"

struct scn_metadata; // capi.cu
namespace scn {
namespace {
template <bool BACKWARD>
__global__ void __launch_bounds__(256) k_sparse_dense(const int *__restrict__ id2pOrP2id, const int4 *__restrict__ coords, int n, int C, long vol, int sy, int sz,
                                                      const float *__restrict__ src, float *__restrict__ dst) {
  __shared__ float tile[32][33];
  __shared__ long s_cell[32]; // dense cell (batch * C * vol + offset) of each site of the tile
  __shared__ int s_row[32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 32 x 8
  const int nTiles = (n + 31) / 32;
  for (int t = blockIdx.x; t < nTiles; t += gridDim.x) {
    const int p = t * 32 + tx;
    if (ty == 0) {
      int row = -1;
      long cell = 0;
      if (p < n) {
        row = id2pOrP2id[p]; // site in spatial order -> feature row
        const int4 c = coords[row];
        cell = (long)c.w * C * vol + ((long)c.x * sy + c.y) * sz + c.z; // RectangularRegion::offset, last dimension fastest
      }
      s_row[tx] = row;
      s_cell[tx] = cell;
    }
    __syncthreads();
    for (int c0 = 0; c0 < C; c0 += 32) {
      if (!BACKWARD) {
        for (int j = ty; j < 32; j += 8) { // site j: 32 consecutive planes
          const int row = s_row[j];
          tile[j][tx] = (row >= 0 && c0 + tx < C) ? __ldg(src + (long)row * C + c0 + tx) : 0.f;
        }
        __syncthreads();
        for (int j = ty; j < 32; j += 8) { // plane c0 + j: 32 sites
          if (c0 + j < C && s_row[tx] >= 0) dst[s_cell[tx] + (long)(c0 + j) * vol] = tile[tx][j];
        }
      } else {
        for (int j = ty; j < 32; j += 8) tile[tx][j] = (c0 + j < C && s_row[tx] >= 0) ? __ldg(src + s_cell[tx] + (long)(c0 + j) * vol) : 0.f;
        __syncthreads();
        for (int j = ty; j < 32; j += 8) {
          const int row = s_row[j];
          if (row >= 0 && c0 + tx < C) dst[(long)row * C + c0 + tx] = tile[j][tx];
        }
      }
      __syncthreads();
    }
  }
}
int run(scn_metadata *m, const long sz[3], const float *src, float *dst, int C, bool backward) {
  Metadata &M = *metadata_of(m);
  Grid *g = M.find_grid(sz);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  SCN_TRY(M.wait_ready(g->rdy));
  cudaStream_t s = M.cstream;
  const long vol = sz[0] * sz[1] * sz[2];
  if (!backward) SCN_CUDA(cudaMemsetAsync(dst, 0, (size_t)g->batch * C * vol * sizeof(float), s)); // output_features.zero_(), CPU/SparseToDense.cpp:46
  if (g->n == 0) return 0;
  const int grid = std::min(cdiv(g->n, 32), kSMs * 8);
  if (backward) k_sparse_dense<true><<<grid, 256, 0, LS(s)>>>(g->p2id, g->coords, g->n, C, vol, (int)sz[1], (int)sz[2], src, dst);
  else k_sparse_dense<false><<<grid, 256, 0, LS(s)>>>(g->p2id, g->coords, g->n, C, vol, (int)sz[1], (int)sz[2], src, dst);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
} // namespace
} // namespace scn

extern "C" {
int scn_sparse_to_dense_forward(scn_metadata *m, const long spatial_size[3], const float *in, float *out, int n_planes) {
  if (!m) { scn::set_error("null scn_metadata handle"); return -3; }
  return scn::run(m, spatial_size, in, out, n_planes, false);
}
int scn_sparse_to_dense_backward(scn_metadata *m, const long spatial_size[3], float *d_in, const float *d_out, int n_planes) {
  if (!m) { scn::set_error("null scn_metadata handle"); return -3; }
  return scn::run(m, spatial_size, d_out, d_in, n_planes, true);
}
}
