"""Fusion requests of the C ABI (scn_fuse_next_lateral / scn_fuse_next_stats) belong to the next call of one of the three
convolution forward entries on the thread -- submanifold, strided, deconvolution -- and to nothing else.  A NetworkInNetwork
forward leaves them pending and computes exactly what it computes without them; a forward entry that cannot honour them (the
CUDA-core path in fp32 mode) still takes them, so they do not reach a later, unrelated call.  scn_debug_counter(3) counts
launches that folded in a lateral stage, scn_debug_counter(4) launches whose epilogue accumulated statistics."""
import ctypes as C

import pytest
import torch

from detection_3d_b200 import synthetic

pytestmark = pytest.mark.gpu
CNT = dict(lateral=3, stats=4, tc=7, simt=10)
# large enough that no launch splits its filter offsets over CTAs (the epilogue statistics need whole work items)
BLD = dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)
FULL = [2048, 2048, 512]
C0 = 64


def _counters(lib):
    return {k: lib.scn_debug_counter(i) for k, i in CNT.items()}


def _delta(lib, before):
    now = _counters(lib)
    return {k: now[k] - before[k] for k in now}


def _setup():
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200._lib import lib
    from gpu_adapter import GpuMetadata
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    G = GpuMetadata()
    n = G.input_layer(FULL, synthetic.building_coords(**BLD), 0, 4)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(n, C0, generator=g).cuda()
    w = (torch.randn(27, 1, C0, C0, generator=g) * 0.05).cuda()
    y = torch.randn(n, C0, generator=g).cuda()
    wl = (torch.randn(C0, C0, generator=g) * 0.05).cuda()
    return scn, lib(), G, n, x, w, y, wl


def _p(t):
    return C.c_void_p(t.data_ptr())


def _subm(lib, G, x, w, out):
    from detection_3d_b200._lib import check, l3
    macs = C.c_double()
    check(lib.scn_submanifold_convolution_forward(G.m._h, l3(FULL), l3([3, 3, 3]), _p(x), _p(out), _p(w), None, C0, C0, C.byref(macs), None, 0,
                                                   None, None))


def _nin(lib, x, w, out, n):
    from detection_3d_b200._lib import check
    macs = C.c_double()
    check(lib.scn_network_in_network_forward(_p(x), _p(out), _p(w), None, n, C0, C0, C.byref(macs), C.c_void_p(torch.cuda.current_stream().cuda_stream),
                                             None, 0))


def _result(lib):
    from detection_3d_b200._lib import check
    took_l, took_s = C.c_int(), C.c_int()
    check(lib.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
    return took_l.value, took_s.value


def test_network_in_network_leaves_requests_to_the_next_convolution():
    """Armed requests pass over a tensor-core NetworkInNetwork forward untouched, and the submanifold forward after it takes both."""
    scn, lib, G, n, x, w, y, wl = _setup()
    from detection_3d_b200._lib import check
    wn = w[13, 0].contiguous()
    stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
    plain, nin, out = (torch.empty(n, C0, device="cuda") for _ in range(3))
    try:
        scn.set_math_mode("tf32")
        _result(lib)  # nothing pending from earlier calls
        _nin(lib, x, wn, plain, n)
        before = _counters(lib)
        check(lib.scn_fuse_next_lateral(_p(y), None, _p(wl), 0, C0, n))
        check(lib.scn_fuse_next_stats(_p(stats)))
        _nin(lib, x, wn, nin, n)
        d_nin = _delta(lib, before)
        before = _counters(lib)
        _subm(lib, G, x, w, out)
        d_subm = _delta(lib, before)
        took = _result(lib)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert d_nin["tc"] == 1 and d_nin["lateral"] == 0 and d_nin["stats"] == 0, d_nin
    assert torch.equal(nin, plain), "an armed request changed the NetworkInNetwork output"
    assert d_subm["tc"] == 1 and d_subm["lateral"] == 1 and d_subm["stats"] == 1, d_subm
    assert took == (1, 1), took
    assert float(stats.abs().sum()) > 0


def test_cuda_core_forward_drops_the_request():
    """A forward on the CUDA cores takes the request it cannot honour: the tensor-core forward after it, not re-armed, accumulates
    no statistics."""
    scn, lib, G, n, x, w, y, wl = _setup()
    from detection_3d_b200._lib import check
    stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
    out = torch.empty(n, C0, device="cuda")
    try:
        scn.set_math_mode("fp32")
        _result(lib)
        check(lib.scn_fuse_next_stats(_p(stats)))
        before = _counters(lib)
        _subm(lib, G, x, w, out)
        d32 = _delta(lib, before)
        scn.set_math_mode("tf32")
        before = _counters(lib)
        _subm(lib, G, x, w, out)
        d = _delta(lib, before)
        took = _result(lib)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert d32["simt"] >= 1 and d32["tc"] == 0 and d32["stats"] == 0, d32
    assert d["tc"] == 1 and d["stats"] == 0, d
    assert took == (0, 0), took
    assert float(stats.abs().sum()) == 0
