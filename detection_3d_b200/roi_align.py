"""ROIAlignRotated3D on the backbone's sparse roi maps (SURVEY.md section 8f rank 3), behind the reference's module interface:
maskrcnn_benchmark/layers/roi_align_rotated_3d.py:56-94 (`ROIAlignRotated3D(output_size, spatial_scale, sampling_ratio)`,
`forward(input_s3d, rois_3d)` -> [n_rois, C, ph, pw, pz]).  The reference densifies the sparse map first
(sparse_3d_to_dense_2d) and samples the dense tensor (csrc/cuda/ROIAlignRotated3D_cuda.cu); here the CUDA kernel samples the
sparse grid directly (detection_3d_b200/csrc/roialign.cu) -- same values, no 268 MB zero fill per call."""
import ctypes as C
import warnings

import torch
from torch import nn
from torch.autograd import Function

from ._lib import check, l3, lib


def _extent(input_s3d):
    """height, width, zsize of the dense tensor the reference would sample: the occupied extent (tools_3d_2d.py:15-17,30)."""
    md, sz = input_s3d.metadata, input_s3d.spatial_size
    loc = md.getSpatialLocations(sz, device="cuda") if hasattr(md, "getSpatialLocations") else input_s3d.get_spatial_locations()
    return [int(v) for v in (loc[:, :3].max(0)[0] + 1).tolist()]


def _alert_not_deterministic(op):
    """torch's convention for an op without a deterministic implementation under torch.use_deterministic_algorithms(True): raise, or
    warn in warn-only mode."""
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f"{op} does not have a deterministic implementation, but you set 'torch.use_deterministic_algorithms(True)'. You can turn off "
           "determinism just for this operation, or you can use the 'warn_only=True' option, if that's acceptable for your application.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg)
    else:
        raise RuntimeError(msg)


class _ROIAlignRotated3D(Function):
    @staticmethod
    def forward(ctx, features, metadata, spatial_size, extent, roi, output_size, spatial_scale, sampling_ratio):
        feats = features.contiguous()
        roi = roi.contiguous().float()
        ctx.save_for_backward(roi)
        ctx.args = (metadata, [int(v) for v in spatial_size.tolist()], extent, tuple(int(v) for v in output_size), float(spatial_scale), int(sampling_ratio),
                    tuple(feats.shape))
        ph, pw, pz = ctx.args[3]
        out = torch.empty((roi.size(0), feats.size(1), ph, pw, pz), dtype=torch.float32, device=feats.device)
        if out.numel():
            check(lib().scn_roi_align_rotated_3d_forward(metadata._h, l3(ctx.args[1]), C.c_void_p(feats.data_ptr()), feats.size(1), (C.c_int * 3)(*extent),
                                                         C.c_void_p(roi.data_ptr()), roi.size(0), ctx.args[4], ph, pw, pz, ctx.args[5], C.c_void_p(out.data_ptr())))
        return out

    @staticmethod
    def backward(ctx, grad_output):
        _alert_not_deterministic("ROIAlignRotated3D backward")  # (gradients are scattered into the feature rows with float atomics)
        roi, = ctx.saved_tensors
        metadata, sz, extent, (ph, pw, pz), scale, sampling, shape = ctx.args
        g = grad_output.contiguous()
        d = torch.empty(shape, dtype=torch.float32, device=g.device)
        if d.numel():
            check(lib().scn_roi_align_rotated_3d_backward(metadata._h, l3(sz), C.c_void_p(d.data_ptr()), shape[1], (C.c_int * 3)(*extent), C.c_void_p(roi.data_ptr()),
                                                          roi.size(0), scale, ph, pw, pz, sampling, C.c_void_p(g.data_ptr())))
        return d, None, None, None, None, None, None, None


class ROIAlignRotated3D(nn.Module):
    def __init__(self, output_size, spatial_scale, sampling_ratio):
        super().__init__()
        self.output_size = output_size
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio

    def forward(self, input_s3d, rois_3d):
        """input_s3d: SparseConvNetTensor (CUDA features); rois_3d: CUDA float [n, 8] = (batch, center_w, center_h, center_z, w, h, z,
        theta in degrees) in the coordinate frame of the dense tensor the reference builds ([B, C, X, Y, Z]: height = X, width = Y)."""
        if not (input_s3d.features.is_cuda and rois_3d.is_cuda):
            raise RuntimeError("ROIAlignRotated3D: expected CUDA tensors (this implementation has no CPU path)")
        fn = _ROIAlignRotated3D.apply if torch.is_grad_enabled() else (lambda *a: _ROIAlignRotated3D.forward(_Ctx(), *a))
        return fn(input_s3d.features, input_s3d.metadata, input_s3d.spatial_size, _extent(input_s3d), rois_3d, self.output_size, self.spatial_scale, self.sampling_ratio)

    def __repr__(self):
        return f"{self.__class__.__name__}(output_size={self.output_size}, spatial_scale={self.spatial_scale}, sampling_ratio={self.sampling_ratio})"


class _Ctx(object):
    def save_for_backward(self, *t):
        pass
