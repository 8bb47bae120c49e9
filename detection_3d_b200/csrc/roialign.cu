// ROIAlignRotated3D straight from the SPARSE feature map.
//   reference: maskrcnn_benchmark/layers/roi_align_rotated_3d.py:56-86 (module: sparse_3d_to_dense_2d -> dense [B, C, X, Y, Z] cropped to
//   the occupied extent -> _C.roi_align_rotated_3d_forward) and maskrcnn_benchmark/csrc/cuda/ROIAlignRotated3D_cuda.cu:16-172 (forward),
//   :176-346 (backward).
// The reference densifies first: for the level-4 roi map of the B470 building that is a 268 MB zero fill and a scatter per call, read
// back at eight corners per sample.  Here every corner is looked up in the sparse grid (block directory + occupancy word, L1 / L2
// resident) and only ACTIVE corners touch feature memory -- an inactive corner is the zero the dense tensor would have held.
// Same arithmetic as the reference kernel: no rounding of the roi, theta in degrees, malformed rois forced to 1 x 1 x 1, sample grid
// = sampling_ratio (or ceil(roi / pooled)) per dimension, trilinear weights with the low / high clamping of bilinear_interpolate
// (including its `zsize > zsize` test, which never rejects a sample for being above the map), average over the samples of a bin.
// Dimension naming follows the reference: height <-> x coordinate of the grid, width <-> y, zsize <-> z; roi = (batch, center_w,
// center_h, center_z, w, h, z, theta).
// One CTA per (roi, ph): its pw x pz bins go warp by warp (lanes over channels, the 8 corners of a sample are computed by lanes 0-7
// and broadcast), results are staged in shared memory and leave as contiguous pw x pz runs of the [n][C][ph][pw][pz] output.
#include "../../include/scn_b200.h"
#include "metadata.cuh"

struct scn_metadata;
namespace scn {
Metadata *metadata_of(scn_metadata *m);
namespace {
struct RoiGeom {
  float cw, ch, cz, w, h, z, cosT, sinT, binH, binW, binZ, startH, startW, startZ;
  int gh, gw, gz, batch;
};
__device__ __forceinline__ RoiGeom roi_geom(const float *r, float scale, int PH, int PW, int PZ, int sampling) {
  RoiGeom g;
  g.batch = (int)r[0];
  g.cw = r[1] * scale; g.ch = r[2] * scale; g.cz = r[3] * scale;
  g.w = fmaxf(r[4] * scale, 1.f); g.h = fmaxf(r[5] * scale, 1.f); g.z = fmaxf(r[6] * scale, 1.f);
  const float theta = (float)(r[7] * M_PI / 180.0); // (the reference evaluates theta in float after a double product, :127)
  g.binH = g.h / (float)PH; g.binW = g.w / (float)PW; g.binZ = g.z / (float)PZ;
  g.gh = sampling > 0 ? sampling : (int)ceilf(g.h / PH);
  g.gw = sampling > 0 ? sampling : (int)ceilf(g.w / PW);
  g.gz = sampling > 0 ? sampling : (int)ceilf(g.z / PZ);
  g.startH = -g.h / 2.0f; g.startW = -g.w / 2.0f; g.startZ = -g.z / 2.0f;
  g.cosT = cosf(theta); g.sinT = sinf(theta);
  return g;
}
// corner j (0..7) of the sample at (y, x, z): grid row (or -1) and trilinear weight; false when the sample lies outside the map
template <bool BACKWARD>
__device__ __forceinline__ bool sample_corner(const GridView &gv, const int *__restrict__ p2id, int H, int W, int Z, float y, float x, float z, int batch, int j,
                                              int &row, float &wgt) {
  row = -1; wgt = 0.f;
  // forward (:27): `zsize > zsize` never rejects a sample above the map (it is clamped to the top layer instead); the gradient
  // variant (:184) does test z > zsize -- the reference's forward and backward disagree there, and so do these two
  if (y < -1.0f || y > H || x < -1.0f || x > W || z < -1.0f || (BACKWARD && z > Z)) return false;
  if (y <= 0) y = 0;
  if (x <= 0) x = 0;
  if (z <= 0) z = 0;
  int yl = (int)y, xl = (int)x, zl = (int)z, yh, xh, zh;
  if (yl >= H - 1) { yh = yl = H - 1; y = (float)yl; } else yh = yl + 1;
  if (xl >= W - 1) { xh = xl = W - 1; x = (float)xl; } else xh = xl + 1;
  if (zl >= Z - 1) { zh = zl = Z - 1; z = (float)zl; } else zh = zl + 1;
  const float ly = y - yl, lx = x - xl, lz = z - zl, hy = 1.f - ly, hx = 1.f - lx, hz = 1.f - lz;
  // corner order of the reference: v1..v4 at z_low = (yl,xl) (yl,xh) (yh,xl) (yh,xh), v5..v8 the same at z_high
  const int yy = (j & 2) ? yh : yl, xx = (j & 1) ? xh : xl, zz = (j & 4) ? zh : zl;
  wgt = ((j & 2) ? ly : hy) * ((j & 1) ? lx : hx) * ((j & 4) ? lz : hz);
  const int p = grid_lookup(gv, yy, xx, zz, batch); // height <-> grid x, width <-> grid y
  row = p >= 0 ? __ldg(p2id + p) : -1;
  return true;
}
template <bool BACKWARD>
__global__ void __launch_bounds__(256) k_roi_align(GridView gv, const int *__restrict__ p2id, const float *__restrict__ feats, float *__restrict__ dFeats, int C, int H,
                                                   int W, int Z, const float *__restrict__ rois, float scale, int PH, int PW, int PZ, int sampling,
                                                   float *__restrict__ out, const float *__restrict__ dOut) {
  extern __shared__ float stage[]; // forward: [min(C, 128)][PW * PZ]
  const int n = blockIdx.x / PH, ph = blockIdx.x % PH;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nWarps = blockDim.x >> 5;
  const RoiGeom g = roi_geom(rois + (long)n * 8, scale, PH, PW, PZ, sampling);
  const float count = (float)(g.gh * g.gw * g.gz);
  const int nBins = PW * PZ;
  for (int c0 = 0; c0 < C; c0 += 128) {
    const int cN = min(128, C - c0);
    for (int b = warp; b < nBins; b += nWarps) {
      const int pw = b / PZ, pz = b % PZ;
      float acc[4] = {0.f, 0.f, 0.f, 0.f}, top[4] = {0.f, 0.f, 0.f, 0.f};
      if (BACKWARD) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int c = c0 + lane + 32 * q;
          if (c < C) top[q] = __ldg(dOut + (((long)n * C + c) * PH + ph) * nBins + b);
        }
      }
      for (int iy = 0; iy < g.gh; iy++) {
        const float yy = g.startH + ph * g.binH + (iy + .5f) * g.binH / (float)g.gh;
        for (int ix = 0; ix < g.gw; ix++) {
          const float xx = g.startW + pw * g.binW + (ix + .5f) * g.binW / (float)g.gw;
          for (int iz = 0; iz < g.gz; iz++) {
            const float zz = g.startZ + pz * g.binZ + (iz + .5f) * g.binZ / (float)g.gz;
            const float x = xx * g.cosT + yy * g.sinT + g.cw, y = yy * g.cosT - xx * g.sinT + g.ch, z = zz + g.cz;
            int row = -1;
            float wgt = 0.f;
            if (lane < 8) sample_corner<BACKWARD>(gv, p2id, H, W, Z, y, x, z, g.batch, lane, row, wgt);
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const int r = __shfl_sync(0xffffffffu, row, j);
              const float w = __shfl_sync(0xffffffffu, wgt, j);
              if (r < 0) continue;
#pragma unroll
              for (int q = 0; q < 4; q++) {
                const int c = c0 + lane + 32 * q;
                if (c >= C) continue;
                if (BACKWARD) atomicAdd(dFeats + (long)r * C + c, top[q] * w / count);
                else acc[q] = fmaf(w, __ldg(feats + (long)r * C + c), acc[q]);
              }
            }
          }
        }
      }
      if (!BACKWARD) {
#pragma unroll
        for (int q = 0; q < 4; q++)
          if (lane + 32 * q < cN) stage[(lane + 32 * q) * nBins + b] = acc[q] / count;
      }
    }
    if (!BACKWARD) {
      __syncthreads();
      for (int i = threadIdx.x; i < cN * nBins; i += blockDim.x) {
        const int c = i / nBins, b = i % nBins;
        out[(((long)n * C + c0 + c) * PH + ph) * nBins + b] = stage[i];
      }
      __syncthreads();
    }
  }
}
int run(scn_metadata *m, const long sz[3], const float *feats, float *dFeats, int C, const int ext[3], const float *rois, long nRois, float scale, int PH, int PW, int PZ,
        int sampling, float *out, const float *dOut, bool backward) {
  Metadata &M = *metadata_of(m);
  Grid *g = M.find_grid(sz);
  SCN_CHECK(g, "no active sites recorded for this spatial size");
  SCN_CHECK(C > 0 && PH > 0 && PW > 0 && PZ > 0 && nRois >= 0 && ext[0] > 0 && ext[1] > 0 && ext[2] > 0, "roi align arguments");
  SCN_TRY(M.wait_ready(g->rdy));
  cudaStream_t s = M.cstream;
  if (backward) SCN_CUDA(cudaMemsetAsync(dFeats, 0, (size_t)g->n * C * sizeof(float), s));
  if (nRois == 0 || g->n == 0) {
    if (!backward && nRois) SCN_CUDA(cudaMemsetAsync(out, 0, (size_t)nRois * C * PH * PW * PZ * sizeof(float), s));
    return 0;
  }
  const GridView v{g->dir, g->bmask, g->wbase, g->dd[0], g->dd[1], g->dd[2], g->dirCells, (int)g->sz[0], (int)g->sz[1], (int)g->sz[2]};
  const size_t smem = backward ? 0 : (size_t)std::min(C, 128) * PW * PZ * sizeof(float);
  SCN_CHECK(smem <= 200 * 1024, "pooled output too large for the staging buffer");
  if (smem > 48 * 1024) SCN_CUDA(cudaFuncSetAttribute(k_roi_align<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)(nRois * PH);
  if (backward) ++g_counters[kCntFloatAtomic]; // (no deterministic variant: the Python layer raises or warns under torch.use_deterministic_algorithms)
  if (backward) k_roi_align<true><<<grid, 256, 0, LS(s)>>>(v, g->p2id, nullptr, dFeats, C, ext[0], ext[1], ext[2], rois, scale, PH, PW, PZ, sampling, nullptr, dOut);
  else k_roi_align<false><<<grid, 256, smem, LS(s)>>>(v, g->p2id, feats, nullptr, C, ext[0], ext[1], ext[2], rois, scale, PH, PW, PZ, sampling, out, nullptr);
  SCN_CUDA(cudaGetLastError());
  return 0;
}
} // namespace
} // namespace scn

extern "C" {
int scn_roi_align_rotated_3d_forward(scn_metadata *m, const long spatial_size[3], const float *feats, int n_planes, const int extent[3], const float *rois,
                                     long n_rois, float spatial_scale, int pooled_h, int pooled_w, int pooled_z, int sampling_ratio, float *out) {
  if (!m) { scn::set_error("null scn_metadata handle"); return -3; }
  return scn::run(m, spatial_size, feats, nullptr, n_planes, extent, rois, n_rois, spatial_scale, pooled_h, pooled_w, pooled_z, sampling_ratio, out, nullptr, false);
}
int scn_roi_align_rotated_3d_backward(scn_metadata *m, const long spatial_size[3], float *d_feats, int n_planes, const int extent[3], const float *rois,
                                      long n_rois, float spatial_scale, int pooled_h, int pooled_w, int pooled_z, int sampling_ratio, const float *d_out) {
  if (!m) { scn::set_error("null scn_metadata handle"); return -3; }
  return scn::run(m, spatial_size, nullptr, d_feats, n_planes, extent, rois, n_rois, spatial_scale, pooled_h, pooled_w, pooled_z, sampling_ratio, nullptr, d_out, true);
}
}
