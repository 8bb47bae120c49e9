"""ctypes binding of the C-ABI library (include/scn_b200.h).

The CUDA extension is the product: if libscn_b200.so is missing or no CUDA device is present the
import of any operator fails loudly -- there is no CPU or PyTorch fallback.
"""
import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libscn_b200.so")

_lib = None
_det = None  # the deterministic-mode flag last handed to the library
L3 = C.c_long * 3

# every symbol include/scn_b200.h declares: (restype, argtypes)
_vp, _l, _i, _f, _d = C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_double
_pl, _pi, _pd = C.POINTER(C.c_long), C.POINTER(C.c_int), C.POINTER(C.c_double)
SYMBOLS = {
    "scn_last_error": (C.c_char_p, []),
    "scn_version": (_i, []),
    "scn_n_rulebook_bits": (_i, []),
    "scn_metadata_create": (_i, [C.POINTER(_vp), _vp]),
    "scn_metadata_destroy": (None, [_vp]),
    "scn_metadata_prefetch": (_i, [_vp, _i, _vp]),
    "scn_program_create": (_i, [C.POINTER(_vp)]),
    "scn_program_destroy": (None, [_vp]),
    "scn_program_add": (_i, [_vp, _i, _vp, _i, _vp, _i]),
    "scn_program_finish": (_i, [_vp, _i, _vp, _i]),
    "scn_program_run": (_i, [_vp, _vp, _vp, _i, _l, _i, _vp, _vp, _vp, _i, _vp, _pd]),
    "scn_program_output": (_i, [_vp, _i, C.POINTER(_l), C.POINTER(_i), C.POINTER(_vp)]),
    "scn_program_prepare": (_i, [_vp, _vp, _vp, _i, _l, _i]),
    "scn_program_throttle": (_i, [_vp]),
    "scn_program_set_training": (_i, [_vp, _i]),
    "scn_program_backward": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _pi, _vp]),
    "scn_metadata_set_internal_numbering": (_i, [_vp, _i]),
    "scn_get_batch_size": (_i, [_vp, L3, _pi]),
    "scn_metadata_build_reference_grids": (_i, [_vp, L3, _vp, _i, _l, _i, _i, _i, _i, _vp, _vp]),
    "scn_metadata_wait_jobs": (_i, [_vp]),
    "scn_rows_to_reference_order": (_i, [_vp, _vp, L3, _vp, _vp, _i]),
    "scn_program_output_copy": (_i, [_vp, _vp, _i, L3, _vp]),
    "scn_program_outputs_copy": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "scn_rows_to_reference_order_multi": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "scn_rows_from_reference_order": (_i, [_vp, _vp, L3, _vp, _vp, _i]),
    "scn_set_pool_growth": (_i, [_i]),
    "scn_input_layer_built": (_i, [_vp, _pl, _pi]),
    "scn_copy_device": (_i, [_vp, _vp, _l, _vp]),
    "scn_input_layer_build": (_i, [_vp, L3, _vp, _i, _l, _i, _i, _i, _pl, _pi]),
    "scn_input_layer_forward": (_i, [_vp, _vp, _vp, _i]),
    "scn_input_layer_forward_padded_bf16": (_i, [_vp, _vp, _vp, _vp, _i, _i]),
    "scn_input_layer_backward": (_i, [_vp, _vp, _vp, _i]),
    "scn_output_layer_forward": (_i, [_vp, _vp, _vp, _i]),
    "scn_output_layer_backward": (_i, [_vp, _vp, _vp, _i]),
    "scn_get_nactive": (_i, [_vp, L3, _pl]),
    "scn_get_spatial_locations": (_i, [_vp, L3, _vp, _i]),
    "scn_submanifold_prepare": (_i, [_vp, L3, L3, _pl]),
    "scn_convolution_prepare": (_i, [_vp, L3, L3, L3, L3, _pl, _pl]),
    "scn_rulebook_info": (_i, [_vp, _i, L3, L3, L3, _pi, _pl]),
    "scn_rulebook_copy": (_i, [_vp, _i, L3, L3, L3, _i, _vp]),
    "scn_iteration_order": (_i, [_vp, L3, _vp]),
    "scn_submanifold_convolution_forward": (_i, [_vp, L3, L3, _vp, _vp, _vp, _vp, _i, _i, _pd, _vp, C.c_longlong, _vp, _vp]),
    "scn_convolution_forward": (_i, [_vp, L3, L3, L3, L3, _vp, _vp, _vp, _vp, _i, _i, _pd, _vp, C.c_longlong, _vp, _vp]),
    "scn_deconvolution_forward": (_i, [_vp, L3, L3, L3, L3, _vp, _vp, _vp, _vp, _i, _i, _pd, _vp, C.c_longlong, _vp, _vp]),
    "scn_submanifold_convolution_backward": (_i, [_vp, L3, L3, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i]),
    "scn_convolution_backward": (_i, [_vp, L3, L3, L3, L3, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i]),
    "scn_deconvolution_backward": (_i, [_vp, L3, L3, L3, L3, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i]),
    "scn_batchnorm_forward": (_i, [_vp, _vp, _l, _i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _f, _vp, _vp]),
    "scn_batchnorm_backward": (_i, [_vp, _vp, _vp, _vp, _l, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp]),
    "scn_network_in_network_forward": (_i, [_vp, _vp, _vp, _vp, _l, _i, _i, _pd, _vp, _vp, C.c_longlong]),
    "scn_network_in_network_backward_input": (_i, [_vp, _vp, _vp, _l, _i, _i, _vp]),
    "scn_network_in_network_backward_params": (_i, [_vp, _vp, _vp, _vp, _l, _i, _i, _vp]),
    "scn_add_features": (_i, [_vp, _vp, _vp, _l, _vp, _vp]),
    "scn_sparse_to_dense_forward": (_i, [_vp, L3, _vp, _vp, _i]),
    "scn_sparse_to_dense_backward": (_i, [_vp, L3, _vp, _vp, _i]),
    "scn_rpn_head_forward": (_i, [_vp, _l, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "scn_rpn_grid_anchors": (_i, [_vp, _l, _f, C.POINTER(_f), _vp, _i, _vp, _vp]),
    "scn_roi_align_rotated_3d_forward": (_i, [_vp, L3, _vp, _i, C.POINTER(_i), _vp, _l, _f, _i, _i, _i, _i, _vp]),
    "scn_roi_align_rotated_3d_backward": (_i, [_vp, L3, _vp, _i, C.POINTER(_i), _vp, _l, _f, _i, _i, _i, _i, _vp]),
    "scn_top_k_descending": (_i, [_vp, _l, _i, _l, _vp, _vp, _vp]),
    "scn_box_decode_3d": (_i, [_vp, _vp, _vp, _l, C.POINTER(_f), _f, _i, _vp, _vp]),
    "scn_boxes_iou_3d": (_i, [_vp, _l, _vp, _l, C.POINTER(_f), _i, _i, _vp, _vp]),
    "scn_rotate_nms_3d": (_i, [_vp, _vp, _l, _l, _l, _f, _vp, _vp, _vp]),
    "scn_voxelize_extent": (_i, [_vp, _l, _pd, _pd, _pd, _vp]),
    "scn_voxelize": (_i, [_vp, _vp, _l, _i, _pd, _pd, _d, _pd, _i, _l, _i, _vp, _vp, _pl, _vp]),
    "scn_set_math_mode": (_i, [_i]),
    "scn_get_math_mode": (_i, []),
    "scn_set_deterministic": (_i, [_i]),
    "scn_get_deterministic": (_i, []),
    "scn_tensor_core_path_available": (_i, []),
    "scn_kernel_launch_count": (_l, []),
    "scn_debug_counter": (_l, [_i]),
    "scn_release_cached_memory": (_l, []),
    "scn_fuse_next_lateral": (_i, [_vp, _vp, _vp, C.c_longlong, _i, _l]),
    "scn_fuse_next_stats": (_i, [_vp]),
    "scn_fuse_result": (_i, [_pi, _pi]),
}


def lib():
    """Load libscn_b200.so (built by detection_3d_b200/csrc/Makefile or __graft_entry__.build()).

    Every native call goes through here, so this is also where torch.are_deterministic_algorithms_enabled() is copied into the
    library (scn_set_deterministic) before the call: torch's flag is the package's only switch for the deterministic mode."""
    global _lib, _det
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                "detection_3d_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)  # AttributeError = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    det = torch.are_deterministic_algorithms_enabled()
    if det is not _det:
        _lib.scn_set_deterministic(int(det))
        _det = det
    return _lib


def check(status):
    if status != 0:
        raise RuntimeError("scn_b200: " + lib().scn_last_error().decode("utf-8", "replace"))


_L3_CACHE = {}


def l3(v):
    """long[3] argument.  Spatial / filter sizes arrive as small CPU LongTensors that live as long as
    the module tree; the converted ctypes array is cached on (object id, version) for those."""
    if hasattr(v, "tolist"):
        key = (id(v), v._version) if hasattr(v, "_version") else None
        hit = _L3_CACHE.get(key) if key else None
        if hit is not None and hit[0] is v:
            return hit[1]
        lst = [int(x) for x in v.tolist()]
    else:
        key, lst = None, [int(x) for x in v]
    if len(lst) != 3:
        raise RuntimeError("this build is specialised for dimension 3 (Metadata_3)")
    arr = L3(*lst)
    if key is not None:
        if len(_L3_CACHE) > 4096:
            _L3_CACHE.clear()
        _L3_CACHE[key] = (v, arr)  # keeps `v` alive, so its id cannot be reused while cached
    return arr
