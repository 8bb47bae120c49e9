"""Math mode 'tf32x3' (scn.set_math_mode, code 3): the tcgen05 gather-GEMM with every fp32 operand split into two exact TF32
values, x = hi + lo, and out += A_hi W_lo + A_lo W_hi + A_hi W_hi in one fp32 accumulator.  The dropped A_lo W_lo term and the
rounding of lo leave ~2^-21 relative error per product, so the mode is held to the FP32 tolerances (DESIGN.md section 7), per
layer against the CPU oracle and the exact fp32 CUDA-core mode, end to end against the reference's outputs.
scn_debug_counter(15) counts the TF32X3 launches and scn_debug_counter(10) the CUDA-core ones: together they show that the
layers really ran on the new path."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import fpn_util
from detection_3d_b200 import synthetic
from oracle import scn_oracle as so

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
L = torch.LongTensor
CNT = dict(lateral=3, stats=4, lateral_fallback=6, tc=7, split=9, simt=10, train_replay=11, float_atomic=14, x3=15)
FP32_RTOL, FP32_ATOL = 2e-4, 2e-5   # per layer: rtol, atol x max|ref| (DESIGN.md section 7, the fp32 rows)
E2E_RTOL, E2E_ATOL = 2e-3, 2e-4     # end to end, as test_fpn_forward_fp32_vs_reference_golden
MINI4_BLD = dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)
MID_BLD = dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)
# "The split is in effect": the error of tf32x3 against the fp32 anchor is at most this fraction of the error of tf32 on the same
# inputs.  The operand analysis alone gives ~2^-21 against ~2^-11 per product; measured on B200 (128 -> 128 3x3x3 on level 0 of the
# 300 x 280 x 40 building) the ratio is ~30.  The rest is fp32 accumulation, not the split: against the fp64 sum of its rounded
# operands (lo * lo dropped) tf32x3 stays within 43 x 2^-24 of the sum of |products|, three MMAs per K step against tf32's one
# (tests/test_gpu_tc_exact.py::test_accumulation_error_bound), and the fp32 mode it is compared with carries its own 8 x 2^-24.
SPLIT_RATIO = 25
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _scn():
    import detection_3d_b200.sparseconvnet as scn
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    return scn


def _counters():
    from detection_3d_b200._lib import lib
    return {k: lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _close(got, want, rtol=FP32_RTOL, atol=FP32_ATOL):
    want = np.asarray(want)
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    np.testing.assert_allclose(np.asarray(got), want, rtol=rtol, atol=atol * scale)


def _rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.abs(got - want).max() / max(1e-30, np.abs(want).max()))


def _levels(big=False):
    from gpu_adapter import GpuMetadata
    if big:
        c, full, coarse = synthetic.building_coords(**MID_BLD), [2048, 2048, 512], [1024, 1024, 256]
    else:
        c, full, coarse = synthetic.small_building(40, 36, 12, 3, seed=4), [64, 64, 32], [32, 32, 16]
    G, O = GpuMetadata(), so.OracleMetadata()
    n = G.input_layer(full, c, 0, 4)
    assert n == O.input_layer(full, c, 0, 4)
    return G, O, full, coarse


def _in_mode(scn, math, fn):
    try:
        scn.set_math_mode(math)
        r = fn()
        torch.cuda.synchronize()
        return r
    finally:
        scn.set_math_mode("fp32")


def _subm(scn, G, sz, x, w, f):
    out = torch.empty(0, device="cuda")
    macs = scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([f] * 3), G.m, x, out, w, torch.Tensor())
    return out, macs


# ------------------------------------------------------------------ the mode itself
def test_math_mode_code_and_range():
    scn = _scn()
    from detection_3d_b200._lib import lib
    try:
        scn.set_math_mode("tf32x3")
        assert scn.SCN.math_mode() == 3 and lib().scn_get_math_mode() == 3
        assert lib().scn_set_math_mode(4) != 0 and lib().scn_get_math_mode() == 3
        assert b"tf32x3" in lib().scn_last_error()
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ per layer, against the oracle and the fp32 mode
@pytest.mark.parametrize("cin,cout,f", [(9, 32, 3), (32, 32, 3), (64, 64, 3), (128, 128, 3), (256, 256, 3), (32, 128, 1), (64, 128, 3),
                                       (256, 128, 1), (20, 64, 3), (48, 256, 3)])
def test_submanifold_forward(cin, cout, f):
    """Small level (<= 40 work items: the filter offsets are split over CTAs).  Narrow and odd input widths run on zero-padded
    fp32 rows; every layer here takes the tensor-core path."""
    scn = _scn()
    G, O, sz, _ = _levels()
    n = O.nactive(sz)
    rs = np.random.RandomState(cin * 3 + cout + f)
    x = rs.randn(n, cin).astype(np.float32)
    w = (rs.randn(f ** 3, 1, cin, cout) * (2.0 / (cin * f ** 3)) ** 0.5).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, O.submanifold_rules(sz, [f] * 3), n)
    xt, wt = T(x), T(w)
    anchor, _ = _in_mode(scn, "fp32", lambda: _subm(scn, G, sz, xt, wt, f))
    before = _counters()
    (out, got), d = _in_mode(scn, "tf32x3", lambda: _subm(scn, G, sz, xt, wt, f)), _delta(before)
    assert got == macs
    assert d["x3"] == 1 and d["tc"] == 1 and d["simt"] == 0, d
    if f == 3:
        assert d["split"] == 1, d
    _close(out.cpu().numpy(), want)
    _close(out.cpu().numpy(), anchor.cpu().numpy())


def test_large_level_and_split_in_effect():
    """Level 0 of the 300 x 280 x 40 building: more super-tiles than SMs, ragged last tile, one CTA per item.  64 -> 64 against the
    oracle; 128 -> 128 against the fp32 anchor, where the error of tf32x3 must be at most 1/SPLIT_RATIO of the error of tf32 on the
    same inputs."""
    scn = _scn()
    G, O, full, _ = _levels(big=True)
    n = O.nactive(full)
    rs = np.random.RandomState(0)
    x = rs.randn(n, 64).astype(np.float32)
    w = (rs.randn(27, 1, 64, 64) * (2.0 / (64 * 27)) ** 0.5).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, O.submanifold_rules(full, [3, 3, 3]), n)
    before = _counters()
    (out, got), d = _in_mode(scn, "tf32x3", lambda: _subm(scn, G, full, T(x), T(w), 3)), _delta(before)
    assert got == macs and d["x3"] == 1 and d["split"] == 0, d
    _close(out.cpu().numpy(), want)

    x = T(rs.randn(n, 128).astype(np.float32))
    w = T((rs.randn(27, 1, 128, 128) * (2.0 / (128 * 27)) ** 0.5).astype(np.float32))
    anchor = _in_mode(scn, "fp32", lambda: _subm(scn, G, full, x, w, 3)[0]).cpu().numpy()
    e_tf32 = _rel(_in_mode(scn, "tf32", lambda: _subm(scn, G, full, x, w, 3)[0]).cpu().numpy(), anchor)
    x3 = _in_mode(scn, "tf32x3", lambda: _subm(scn, G, full, x, w, 3)[0]).cpu().numpy()
    e_x3 = _rel(x3, anchor)
    print(f"[tf32x3] 128 -> 128 on level 0: max|d| / max|fp32| tf32 {e_tf32:.3e}, tf32x3 {e_x3:.3e} (ratio {e_tf32 / max(e_x3, 1e-30):.0f})")
    assert e_x3 <= e_tf32 / SPLIT_RATIO, (e_x3, e_tf32)
    _close(x3, anchor)


@pytest.mark.parametrize("cin,cout", [(32, 64), (128, 128)])
def test_strided_conv_deconv_and_z_collapse(cin, cout):
    scn = _scn()
    G, O, a, b = _levels()
    f, s = [2, 2, 2], [2, 2, 2]
    rules = O.conv_rules(a, b, f, s)
    rs = np.random.RandomState(cin + cout + 1)
    x = rs.randn(O.nactive(a), cin).astype(np.float32)
    w = (rs.randn(8, 1, cin, cout) * (2.0 / (cin * 8)) ** 0.5).astype(np.float32)
    want, _ = so.o_conv_forward(x, w, rules, O.nactive(b))
    o, fz = [32, 32, 1], [1, 1, 16]
    rz = O.conv_rules(b, o, fz, [1, 1, 1])
    xz = rs.randn(O.nactive(b), cin).astype(np.float32)
    wz = (rs.randn(16, 1, cin, cout) * 0.05).astype(np.float32)
    wantz, _ = so.o_conv_forward(xz, wz, rz, O.nactive(o))
    xd = rs.randn(O.nactive(b), cin).astype(np.float32)
    wantd, macsd = so.o_conv_forward(xd, w, rules, O.nactive(a), deconv=True)

    def run():
        out, outz, outd = torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        scn.SCN.Convolution_updateOutput(L(a), L(b), L(f), L(s), G.m, T(x), out, T(w), torch.Tensor())
        scn.SCN.Convolution_updateOutput(L(b), L(o), L(fz), L([1, 1, 1]), G.m, T(xz), outz, T(wz), torch.Tensor())
        gotd = scn.SCN.Deconvolution_updateOutput(L(b), L(a), L(f), L(s), G.m, T(xd), outd, T(w), torch.Tensor())  # per-offset tile plan
        return out, outz, outd, gotd
    before = _counters()
    (out, outz, outd, gotd), d = _in_mode(scn, "tf32x3", run), _delta(before)
    assert d["x3"] == 3 and d["simt"] == 0, d
    _close(out.cpu().numpy(), want)
    _close(outz.cpu().numpy(), wantz)
    assert gotd == macsd and outd.shape == (O.nactive(a), cout)
    _close(outd.cpu().numpy(), wantd)


def test_network_in_network():
    scn = _scn()
    rs = np.random.RandomState(5)
    x = rs.randn(3000, 64).astype(np.float32)
    w = (rs.randn(64, 128) * 0.1).astype(np.float32)
    b = (rs.randn(128) * 0.1).astype(np.float32)
    want, _ = so.o_nin_forward(x, w)
    out = torch.empty(0, device="cuda")
    before = _counters()
    _in_mode(scn, "tf32x3", lambda: scn.SCN.NetworkInNetwork_updateOutput(T(x), out, T(w), T(b)))
    assert _delta(before)["x3"] == 1
    _close(out.cpu().numpy(), want + b)


def _stats_buffer():
    return torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")


@pytest.mark.parametrize("kind,big,c_lat", [("subm", True, 64), ("subm", True, 32), ("deconv", False, 128), ("deconv", True, 64), ("conv", False, 256)])
def test_lateral_stage_and_epilogue_stats(kind, big, c_lat):
    """out = conv(x) + y[row] @ W_lat in one launch (the lateral rows split like the main ones), with the epilogue BatchNorm
    statistics where the level does not split the filter offsets."""
    scn = _scn()
    from detection_3d_b200._lib import check, l3, lib
    G, O, full, coarse = _levels(big)
    n = O.nactive(full)
    rules2 = O.conv_rules(full, coarse, [2, 2, 2], [2, 2, 2])
    G.conv_rules(full, coarse, [2, 2, 2], [2, 2, 2])
    nc = O.nactive(coarse)
    rs = np.random.RandomState(c_lat + n % 97)
    C0 = 128
    if kind == "subm":
        x = rs.randn(n, C0).astype(np.float32)
        w = (rs.randn(27, 1, C0, C0) * (2.0 / (C0 * 27)) ** 0.5).astype(np.float32)
        conv_out, _ = so.o_conv_forward(x, w, O.submanifold_rules(full, [3, 3, 3]), n)
        n_out = n
    elif kind == "deconv":
        x = rs.randn(nc, C0).astype(np.float32)
        w = (rs.randn(8, 1, C0, C0) * (2.0 / (C0 * 8)) ** 0.5).astype(np.float32)
        conv_out, _ = so.o_conv_forward(x, w, rules2, n, deconv=True)
        n_out = n
    else:
        x = rs.randn(n, C0).astype(np.float32)
        w = (rs.randn(8, 1, C0, C0) * (2.0 / (C0 * 8)) ** 0.5).astype(np.float32)
        conv_out, _ = so.o_conv_forward(x, w, rules2, nc)
        n_out = nc
    y = rs.randn(n_out, c_lat).astype(np.float32)
    wl = (rs.randn(c_lat, C0) * (2.0 / c_lat) ** 0.5).astype(np.float32)
    lat, _ = so.o_nin_forward(y, wl)
    want = conv_out + lat
    p = lambda t: C.c_void_p(t.data_ptr())
    xt, wt, yt, wlt = T(x), T(w), T(y), T(wl)
    out = torch.empty(n_out, C0, device="cuda")
    stats = _stats_buffer()
    macs = C.c_double()
    took_l, took_s = C.c_int(), C.c_int()

    def run():
        check(lib().scn_fuse_next_lateral(p(yt), None, p(wlt), 0, c_lat, n_out))
        check(lib().scn_fuse_next_stats(p(stats)))
        if kind == "subm":
            check(lib().scn_submanifold_convolution_forward(G.m._h, l3(full), l3([3, 3, 3]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        elif kind == "deconv":
            check(lib().scn_deconvolution_forward(G.m._h, l3(coarse), l3(full), l3([2, 2, 2]), l3([2, 2, 2]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        else:
            check(lib().scn_convolution_forward(G.m._h, l3(full), l3(coarse), l3([2, 2, 2]), l3([2, 2, 2]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        check(lib().scn_fuse_result(C.byref(took_l), C.byref(took_s)))
    before = _counters()
    _in_mode(scn, "tf32x3", run)
    d = _delta(before)
    assert took_l.value == 1 and d["lateral"] == 1 and d["x3"] == 1, (took_l.value, d)
    _close(out.cpu().numpy(), want)
    if d["split"] == 0:
        assert took_s.value == 1 and d["stats"] == 1, (took_s.value, d)
        s = stats.view(8, 2, 128).sum(0).cpu().numpy()
        o64 = out.double()
        np.testing.assert_allclose(s[0], o64.sum(0).cpu().numpy(), rtol=1e-4, atol=1e-3 * n_out ** 0.5)
        np.testing.assert_allclose(s[1], (o64 * o64).sum(0).cpu().numpy(), rtol=1e-4)
    else:
        assert took_s.value == 0


@pytest.mark.parametrize("big", [False, True])
def test_fused_epilogue_add(big):
    """out = conv(in) + add_in in the epilogue, against the unfused conv + add, and against the oracle."""
    scn = _scn()
    from detection_3d_b200._lib import check, l3, lib
    G, O, sz, _ = _levels(big)
    n = O.nactive(sz)
    rs = np.random.RandomState(7)
    x, r = rs.randn(n, 64).astype(np.float32), rs.randn(n, 128).astype(np.float32)
    w = (rs.randn(27, 1, 64, 128) * 0.03).astype(np.float32)
    xt, wt, rt = T(x), T(w), T(r)
    p = lambda t: C.c_void_p(t.data_ptr())
    fused = torch.empty(n, 128, device="cuda")

    def run():
        plain, _ = _subm(scn, G, sz, xt, wt, 3)
        macs = C.c_double()
        check(lib().scn_submanifold_convolution_forward(G.m._h, l3(sz), l3([3, 3, 3]), p(xt), p(fused), p(wt), None, 64, 128, C.byref(macs), None,
                                                        C.c_longlong(0), p(rt), None))
        return scn.SCN.add_features(plain, rt)
    want = _in_mode(scn, "tf32x3", run)
    scale = max(1.0, float(want.abs().max()))
    assert float((fused - want).abs().max()) <= 1e-5 * scale  # same products; only the order of the atomic sums may differ
    if not big:
        ref, _ = so.o_conv_forward(x, w, O.submanifold_rules(sz, [3, 3, 3]), n)
        _close(fused.cpu().numpy(), ref + r)


def test_input_gradients():
    """The input gradient of all three convolution kinds runs on the TF32X3 forward kernel with the transposed (and, for the
    submanifold plan, offset-reversed) split weight images; the weight gradient stays on the exact CUDA-core kernel.  The input
    gradient of a 9-channel input (9 output channels of the transposed problem) is one the tensor-core kernel does not take: it
    runs on the CUDA cores, as in tf32 mode."""
    scn = _scn()
    G, O, sz, _ = _levels()
    n = O.nactive(sz)

    def check_grads(din, dw, din_w, dw_w):
        _close(din.cpu().numpy(), din_w)
        _close(dw.cpu().numpy(), dw_w, rtol=1e-3, atol=1e-4)  # (the CUDA-core weight gradient, as in the fp32 parity tests)

    def run():
        for cin, cout, f in [(64, 128, 3), (128, 128, 3), (32, 32, 3), (32, 128, 1), (256, 64, 3), (9, 32, 3)]:
            rs = np.random.RandomState(cin + 3 * cout + f)
            x, dy = rs.randn(n, cin).astype(np.float32), rs.randn(n, cout).astype(np.float32)
            w = (rs.randn(f ** 3, 1, cin, cout) * (2.0 / (cin * f ** 3)) ** 0.5).astype(np.float32)
            din_w, dw_w = so.o_conv_backward(x, dy, w, O.submanifold_rules(sz, [f] * 3))
            out = torch.empty(0, device="cuda")
            scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([f] * 3), G.m, T(x), out, T(w), torch.Tensor())
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            before = _counters()
            scn.SCN.SubmanifoldConvolution_backward(L(sz), L([f] * 3), G.m, T(x), din, T(dy), T(w), dw, torch.Tensor())
            d = _delta(before)
            assert d["x3"] == (1 if cin % 32 == 0 else 0) and (d["simt"] > 0) == (cin % 32 != 0), (cin, d)
            check_grads(din, dw, din_w, dw_w)
        a, b, f, s = [64, 64, 32], [32, 32, 16], [2, 2, 2], [2, 2, 2]
        rules = O.conv_rules(a, b, f, s)
        na, nb = O.nactive(a), O.nactive(b)
        for cin, cout in [(32, 64), (128, 128)]:
            rs = np.random.RandomState(cin + cout)
            x, dy = rs.randn(na, cin).astype(np.float32), rs.randn(nb, cout).astype(np.float32)
            w = (rs.randn(8, 1, cin, cout) * (2.0 / (cin * 8)) ** 0.5).astype(np.float32)
            out = torch.empty(0, device="cuda")
            scn.SCN.Convolution_updateOutput(L(a), L(b), L(f), L(s), G.m, T(x), out, T(w), torch.Tensor())
            din_w, dw_w = so.o_conv_backward(x, dy, w, rules)
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            before = _counters()
            scn.SCN.Convolution_backward(L(a), L(b), L(f), L(s), G.m, T(x), din, T(dy), T(w), dw, torch.Tensor())
            assert _delta(before)["x3"] == 1
            check_grads(din, dw, din_w, dw_w)
            xc, dyf = rs.randn(nb, cin).astype(np.float32), rs.randn(na, cout).astype(np.float32)
            out = torch.empty(0, device="cuda")
            scn.SCN.Deconvolution_updateOutput(L(b), L(a), L(f), L(s), G.m, T(xc), out, T(w), torch.Tensor())
            din_w, dw_w = so.o_conv_backward(xc, dyf, w, rules, deconv=True)
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            before = _counters()
            scn.SCN.Deconvolution_backward(L(b), L(a), L(f), L(s), G.m, T(xc), din, T(dyf), T(w), dw, torch.Tensor())
            assert _delta(before)["x3"] == 1
            check_grads(din, dw, din_w, dw_w)
    _in_mode(scn, "tf32x3", run)


def test_modes_switch_back_and_forth():
    """tf32x3 -> tf32 -> tf32x3 with one weight tensor: each mode keeps its own cached operand image under the tensor's tag (the
    second tf32x3 call gives bit for bit the first one's result, the tf32 call the tf32 error), and an in-place update of the
    weights is seen by the next tf32x3 call."""
    scn = _scn()
    G, O, full, _ = _levels(big=True)
    n = O.nactive(full)
    rs = np.random.RandomState(3)
    x = T(rs.randn(n, 128).astype(np.float32))
    w = T((rs.randn(27, 1, 128, 128) * (2.0 / (128 * 27)) ** 0.5).astype(np.float32))
    conv = lambda: _subm(scn, G, full, x, w, 3)[0]
    anchor = _in_mode(scn, "fp32", conv).cpu().numpy()
    a = _in_mode(scn, "tf32x3", conv)
    t = _in_mode(scn, "tf32", conv)
    b = _in_mode(scn, "tf32x3", conv)
    assert torch.equal(a, b)  # (level 0: one CTA per item, no atomics)
    e_a, e_t = _rel(a.cpu().numpy(), anchor), _rel(t.cpu().numpy(), anchor)
    assert e_a <= e_t / SPLIT_RATIO, (e_a, e_t)
    with torch.no_grad():
        w.mul_(-0.5)
    c = _in_mode(scn, "tf32x3", conv)
    anchor2 = _in_mode(scn, "fp32", conv).cpu().numpy()
    _close(c.cpu().numpy(), anchor2)
    _close(c.cpu().numpy(), -0.5 * a.cpu().numpy())


# ------------------------------------------------------------------ whole network
def _fpn(scn, cfg, seed=1, train=False):
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=seed))
    return net.cuda().train() if train else net.cuda().eval()


def _check_golden(rpn, roi, g):
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        assert len(maps) == int(g[f"n_{tag}"])
        for i, m in enumerate(maps):
            assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
            _close(m.features.cpu().numpy(), g[f"{tag}{i}_features"], rtol=E2E_RTOL, atol=E2E_ATOL)


@pytest.mark.parametrize("name,cfgname,bld", [("mini4", "mini4", MINI4_BLD), ("sw4c_mid", "sw4c", MID_BLD)])
def test_fpn_forward_layerwise_and_replayed_vs_reference_golden(name, cfgname, bld):
    """Layer-by-layer (recording) forward and two replays against the reference's own scn.FPN_Net outputs at the fp32 end-to-end
    tolerances.  A replay launches exactly as many CUDA-core convolutions as a tf32 replay (layers the tensor-core kernel does not
    take: none on the sw4c backbone, whose 8 top-down lateral shortcuts are folded into their deconvolutions); every other
    convolution runs on the TF32X3 kernel."""
    scn = _scn()
    cfg = fpn_util.mini4_config() if cfgname == "mini4" else scn.sw4c_fpn432_config()
    g = np.load(os.path.join(GOLD, f"fpn_{name}.npz"))
    coords = synthetic.building_coords(**bld)
    c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()
    try:
        scn.set_math_mode("tf32")
        with torch.no_grad():
            tnet = _fpn(scn, cfg)
            tnet([c, f])  # records
            before = _counters()
            tnet([c, f])  # replays
            torch.cuda.synchronize()
            simt_tf32 = _delta(before)["simt"]
        scn.set_math_mode("tf32x3")
        net = _fpn(scn, cfg)
        with torch.no_grad():
            before = _counters()
            scn.forward_pass_multiplyAdd_count = 0
            rpn, roi = net([c, f])  # records (layer by layer)
            torch.cuda.synchronize()
            assert _delta(before)["x3"] > 0
            assert scn.forward_pass_multiplyAdd_count == float(g["macs"])
            _check_golden(rpn, roi, g)
            assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
            for rep in range(2):
                before = _counters()
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])  # replays
                torch.cuda.synchronize()
                d = _delta(before)
                assert scn.forward_pass_multiplyAdd_count == float(g["macs"])
                assert d["x3"] > 0 and d["x3"] == d["tc"] and d["simt"] == simt_tf32, (d, simt_tf32)
                if cfgname == "sw4c":
                    assert d["simt"] == 0 and d["lateral"] == 8 and d["lateral_fallback"] == 0, d
                _check_golden(rpn, roi, g)
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.parametrize("replay", [False, True])
def test_training_step_vs_reference_autograd(replay):
    """The whole mini4 training step (tests/golden/fpn_mini4_train.npz) at the fp32-mode bounds of
    test_whole_network_training_step_vs_reference_autograd.  replay=True: the second step, one autograd node
    (scn_program_run in training mode + scn_program_backward)."""
    scn = _scn()
    g = np.load(os.path.join(GOLD, "fpn_mini4_train.npz"))
    tol_max, tol_rms, tol_cos, tol = 5e-3, 5e-3, 0.99999, 5e-3
    coords = synthetic.building_coords(**MINI4_BLD)
    inp = lambda: [torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()]
    try:
        scn.set_math_mode("tf32x3")
        net = _fpn(scn, dict(fpn_util.mini4_config(), track_running_stats=True), train=True)
        if replay:
            rpn, roi = net(inp())
            sum((m.features ** 2).mean() for m in rpn + roi).backward()
            assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
            net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
            net.zero_grad(set_to_none=True)
        before = _counters()
        rpn, roi = net(inp())
        terms = [(m.features ** 2).mean() for m in rpn + roi]
        loss = sum(terms)
        loss.backward()
        torch.cuda.synchronize()
        d = _delta(before)
    finally:
        scn.set_math_mode("fp32")
    assert d["x3"] > 0 and d["train_replay"] == (1 if replay else 0), d
    np.testing.assert_allclose(np.array([float(t.detach()) for t in terms]), g["map_mean_sq"], rtol=tol)
    assert abs(float(loss) - float(g["loss"])) <= tol * float(g["loss"])
    want_keys = {k[5:] for k in g.files if k.startswith("grad:")}
    got = {k: p.grad for k, p in net.named_parameters()}
    assert {k for k, v in got.items() if v is not None} == want_keys
    worst = 0.0
    for k in want_keys:
        ref = g["grad:" + k].astype(np.float64)
        dd = got[k].cpu().numpy().astype(np.float64) - ref
        err = float(np.abs(dd).max() / max(1e-6, np.abs(ref).max()))
        rms = float(np.sqrt((dd * dd).mean()) / max(1e-12, np.sqrt((ref * ref).mean())))
        worst = max(worst, err)
        assert err < tol_max and rms < tol_rms, (k, err, rms)
    keys = sorted(want_keys)
    a = np.concatenate([got[k].cpu().numpy().ravel() for k in keys]).astype(np.float64)
    b = np.concatenate([g["grad:" + k].ravel() for k in keys]).astype(np.float64)
    cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)))
    print(f"[tf32x3] training step (replay={replay}): worst gradient error {worst:.3e} of max|grad|, cosine {cos:.8f}")
    assert cos >= tol_cos, cos
    for k, buf in net.named_buffers():
        ref = g["buf:" + k]
        np.testing.assert_allclose(buf.cpu().numpy(), ref, rtol=tol, atol=tol * max(1e-3, float(np.abs(ref).max())), err_msg=k)


# ------------------------------------------------------------------ deterministic mode
@pytest.fixture
def det():
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn)


def _equal(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and torch.equal(x, y), (i, float((x - y).abs().max()) if x.shape == y.shape else None)


def test_deterministic_mode(det):
    """Under torch.use_deterministic_algorithms(True): two recording forwards of two fresh networks, two replays and two replayed
    training steps are bitwise equal, and no launch accumulated floats with atomics."""
    scn = _scn()
    coords = synthetic.building_coords(**MINI4_BLD)
    c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()

    def forward(net):
        with torch.no_grad():
            rpn, roi = net([c, f])
        return [m.features.clone() for m in rpn + roi]

    def step(net, state):
        net.load_state_dict(state)
        net.zero_grad(set_to_none=True)
        x = f.detach().clone().requires_grad_(True)
        rpn, roi = net([c, x])
        terms = [(m.features ** 2).mean() for m in rpn + roi]
        sum(terms).backward()
        torch.cuda.synchronize()
        return ([t.detach() for t in terms] + [p.grad.clone() for _, p in sorted(net.named_parameters()) if p.grad is not None]
                + [x.grad.clone()] + [b.clone() for _, b in sorted(net.named_buffers())])
    try:
        scn.set_math_mode("tf32x3")
        before = _counters()
        a, b = _fpn(scn, fpn_util.mini4_config()), _fpn(scn, fpn_util.mini4_config())
        _equal(forward(a), forward(b))              # recording forwards
        _equal(forward(a), forward(a))              # replays
        tnet = _fpn(scn, dict(fpn_util.mini4_config(), track_running_stats=True), train=True)
        state = {k: v.clone() for k, v in tnet.state_dict().items()}
        step(tnet, state)                           # records
        assert tnet.__dict__.get("_program_train") is not None, tnet.__dict__.get("_program_train_error")
        _equal(step(tnet, state), step(tnet, state))  # replayed training steps
        d = _delta(before)
    finally:
        scn.set_math_mode("fp32")
    assert d["float_atomic"] == 0 and d["x3"] > 0 and d["split"] > 0, d
