"""GPU parity tests that pin the BENCHMARKED code path (bf16 / tf32 operands, replayed program on an internally numbered
Metadata, lateral 1x1x1 stage folded into the convolution, BatchNorm statistics in the epilogue, bf16-only outputs, packed
narrow rows) to the outputs of the reference itself, plus the pieces round 1 left untested: InputLayer backward, OutputLayer,
NetworkInNetwork, a whole-network training step against the reference's autograd, odd channel counts on the scratch path.
`scn_debug_counter` deltas prove that the fused paths really ran (no silent fallback)."""
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
CNT = dict(lateral=3, stats=4, half_only=5, lateral_fallback=6, tc=7, bn_from_sums=8, split=9, simt=10)

TF32_TOL, BF16_TOL = (4e-3, 2e-3), (1.6e-2, 8e-3)   # per layer: rtol, atol x max|ref|  (operand rounding 2^-10 / 2^-8 per product)
TC_TOL = {"tf32": TF32_TOL, "bf16": BF16_TOL}
TC_E2E = {"tf32": 1e-2, "bf16": 4.5e-2}               # end to end: max |got - ref| / max(1, max|ref|) per returned map


def _scn():
    import detection_3d_b200.sparseconvnet as scn
    return scn


def _counters():
    from detection_3d_b200._lib import lib
    return {k: lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _tc_or_skip(scn):
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")


def _close(got, want, rtol, atol):
    want = np.asarray(want)
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    np.testing.assert_allclose(np.asarray(got), want, rtol=rtol, atol=atol * scale)


def _gpu():
    from gpu_adapter import GpuMetadata
    return GpuMetadata()


T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------ IO layers
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_input_layer_backward_and_output_layer(mode):
    """scn_input_layer_backward vs InputLayer_BackwardPass (SCN/CPU/IOLayers.cpp:30-47,76-95) and the OutputLayer pair
    (:97-140), all five input modes, duplicates present for modes 1-4."""
    scn = _scn()
    rs = np.random.RandomState(40 + mode)
    c = rs.randint(0, 10, (2500, 3))
    if mode == 0:
        c = np.unique(c, axis=0)
        c = c[rs.permutation(c.shape[0])]
    f = rs.randn(c.shape[0], 9).astype(np.float32)
    G, O = _gpu(), so.OracleMetadata()
    n = G.input_layer([16, 16, 16], c, 0, mode, feats=f)
    assert n == O.input_layer([16, 16, 16], c, 0, mode)
    hdr, tab = (O.input_rules() + [np.zeros(0, np.int32)])[:2]
    if mode == 0:
        hdr = np.array([0, 1, c.shape[0], c.shape[0]])
    dy = rs.randn(n, 9).astype(np.float32)
    want = dy.copy() if mode == 0 else so.o_input_layer_backward(dy, hdr, tab)
    din = torch.empty(0, device="cuda")
    scn.SCN.InputLayer_updateGradInput(G.m, din, T(dy))
    assert din.shape == want.shape
    np.testing.assert_allclose(din.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    # OutputLayer forward: voxel rows back to input rows; backward: sums per voxel
    x = rs.randn(n, 5).astype(np.float32)
    out = torch.empty(0, device="cuda")
    scn.SCN.OutputLayer_updateOutput(G.m, T(x), out)
    np.testing.assert_allclose(out.cpu().numpy(), so.o_output_layer_forward(x, hdr, tab), rtol=1e-6, atol=1e-6)
    g = rs.randn(*out.shape).astype(np.float32)
    gin = torch.empty(0, device="cuda")
    scn.SCN.OutputLayer_updateGradInput(G.m, gin, T(g))
    np.testing.assert_allclose(gin.cpu().numpy(), so.o_output_layer_backward(g, hdr, tab), rtol=1e-5, atol=1e-5)


def test_output_layer_module_autograd():
    """scn.OutputLayer through the module API, gradient through InputLayer -> OutputLayer (mode 4): d feats = mean over the voxel."""
    scn = _scn()
    rs = np.random.RandomState(3)
    c = rs.randint(0, 6, (400, 3))
    f = torch.from_numpy(rs.randn(400, 4).astype(np.float32)).cuda().requires_grad_(True)
    inp = scn.InputLayer(3, [8, 8, 8], mode=4)
    x = inp([torch.from_numpy(c), f])
    y = scn.OutputLayer(3)(x)
    assert y.shape == (400, 4)
    w = torch.from_numpy(rs.randn(400, 4).astype(np.float32)).cuda()
    (y * w).sum().backward()
    O = so.OracleMetadata()
    O.input_layer([8, 8, 8], c, 0, 4)
    hdr, tab = O.input_rules()
    want = so.o_input_layer_backward(so.o_output_layer_backward(w.cpu().numpy(), hdr, tab), hdr, tab)
    np.testing.assert_allclose(f.grad.cpu().numpy(), want, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(y.detach().cpu().numpy(), so.o_output_layer_forward(so.o_input_layer_forward(f.detach().cpu().numpy(), hdr, tab), hdr, tab), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ NetworkInNetwork
@pytest.mark.parametrize("math", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("n,cin,cout,bias", [(3000, 64, 128, False), (777, 32, 32, True), (20000, 128, 64, False), (5, 9, 16, True), (0, 32, 32, False)])
def test_network_in_network(math, n, cin, cout, bias):
    """scn.NetworkInNetwork forward + autograd backward vs cpu_NetworkInNetwork_* (SCN/CPU/NetworkInNetwork.cpp:7-46)."""
    scn = _scn()
    if math != "fp32":
        _tc_or_skip(scn)
    rs = np.random.RandomState(n + cin + cout)
    x = rs.randn(n, cin).astype(np.float32)
    dy = rs.randn(n, cout).astype(np.float32)
    rtol, atol = (2e-4, 2e-5) if math == "fp32" else TC_TOL[math]
    try:
        scn.set_math_mode(math)
        m = scn.NetworkInNetwork(cin, cout, bias).cuda()
        if bias:
            with torch.no_grad():
                m.bias.copy_(torch.from_numpy(rs.randn(cout).astype(np.float32)))
        w = m.weight.detach().cpu().numpy()
        b = m.bias.detach().cpu().numpy() if bias else None
        xt = T(x).requires_grad_(True)
        t = scn.SparseConvNetTensor(features=xt, metadata=None, spatial_size=L([8, 8, 8]))
        scn.forward_pass_multiplyAdd_count = 0
        y = m(t).features
        want, macs = so.o_nin_forward(x, w, b)
        assert scn.forward_pass_multiplyAdd_count == macs and y.shape == (n, cout)
        _close(y.detach().cpu().numpy(), want, rtol, atol)
        if n:
            y.backward(T(dy))
            din, dw, db = so.o_nin_backward(x, dy, w)
            _close(xt.grad.cpu().numpy(), din, rtol, atol)
            _close(m.weight.grad.cpu().numpy(), dw, 1e-3, 1e-4)   # weight gradient always runs in fp32 on the CUDA cores
            if bias:
                _close(m.bias.grad.cpu().numpy(), db, 1e-3, 1e-4)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ fused lateral stage and epilogue statistics (C-ABI)
def _stats_buffer():
    return torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")


def _reduce_stats(buf, c):
    s = buf.view(8, 2, 128).sum(0).cpu().numpy()
    return s[0, :c], s[1, :c]


@pytest.mark.parametrize("math", ["tf32", "bf16"])
@pytest.mark.parametrize("kind,big,c_lat", [("subm", True, 64), ("subm", True, 32), ("deconv", False, 128), ("deconv", True, 64), ("conv", False, 256)])
def test_fused_lateral_stage_and_epilogue_stats(math, kind, big, c_lat):
    """out = conv(x) + y[row] @ W_lat with the per-channel sum / sum of squares of `out` accumulated by the epilogue, requested
    through scn_fuse_next_lateral / scn_fuse_next_stats -- the in2 / wimg2 / stats arguments of conv_plan_tc that the replayed
    program uses for the FPN's top-down step.  Checked against the oracle's conv (+ deconv) + NetworkInNetwork + add and
    against out.sum(0), (out * out).sum(0); scn_fuse_result must report that both requests were honoured."""
    scn = _scn()
    from detection_3d_b200._lib import check, l3, lib
    _tc_or_skip(scn)
    if big:
        c = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
        full, coarse = [2048, 2048, 512], [1024, 1024, 256]
    else:
        c = synthetic.small_building(40, 36, 12, 3, seed=4)
        full, coarse = [64, 64, 32], [32, 32, 16]
    G, O = _gpu(), so.OracleMetadata()
    n = G.input_layer(full, c, 0, 4)
    assert n == O.input_layer(full, c, 0, 4)
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
    try:
        scn.set_math_mode(math)
        xt, wt, yt, wlt = T(x), T(w), T(y), T(wl)
        y16 = yt.to(torch.bfloat16)
        out = torch.empty(n_out, C0, device="cuda")
        stats = _stats_buffer()
        macs = C.c_double()
        before = _counters()
        check(lib().scn_fuse_next_lateral(p(yt), p(y16), p(wlt), 0, c_lat, n_out))
        check(lib().scn_fuse_next_stats(p(stats)))
        if kind == "subm":
            check(lib().scn_submanifold_convolution_forward(G.m._h, l3(full), l3([3, 3, 3]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        elif kind == "deconv":
            check(lib().scn_deconvolution_forward(G.m._h, l3(coarse), l3(full), l3([2, 2, 2]), l3([2, 2, 2]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        else:
            check(lib().scn_convolution_forward(G.m._h, l3(full), l3(coarse), l3([2, 2, 2]), l3([2, 2, 2]), p(xt), p(out), p(wt), None, C0, C0, C.byref(macs), None, 0, None, None))
        took_l, took_s = C.c_int(), C.c_int()
        check(lib().scn_fuse_result(C.byref(took_l), C.byref(took_s)))
        torch.cuda.synchronize()
        d = _delta(before)
    finally:
        scn.set_math_mode("fp32")
    assert took_l.value == 1 and d["lateral"] == 1, (took_l.value, d)
    rtol, atol = TC_TOL[math]
    _close(out.cpu().numpy(), want, rtol, atol * 1.5)  # two operand-rounded products summed
    if d["split"] == 0:  # (small levels split the filter offsets over CTAs: no statistics there, by design)
        assert took_s.value == 1 and d["stats"] == 1, (took_s.value, d)
        s1, s2 = _reduce_stats(stats, C0)
        o64 = out.double()
        np.testing.assert_allclose(s1, o64.sum(0).cpu().numpy(), rtol=1e-4, atol=1e-3 * n_out ** 0.5)
        np.testing.assert_allclose(s2, (o64 * o64).sum(0).cpu().numpy(), rtol=1e-4)
    else:
        assert took_s.value == 0


@pytest.mark.parametrize("math", ["tf32", "bf16"])
def test_epilogue_stats_alone_packed_and_plain(math):
    """Statistics request without a lateral on a 32-channel layer (packed rows in bf16 mode) and a 64-channel one."""
    scn = _scn()
    from detection_3d_b200._lib import check, l3, lib
    _tc_or_skip(scn)
    c = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
    full = [2048, 2048, 512]
    G, O = _gpu(), so.OracleMetadata()
    n = G.input_layer(full, c, 0, 4)
    O.input_layer(full, c, 0, 4)
    rules = O.submanifold_rules(full, [3, 3, 3])
    p = lambda t: C.c_void_p(t.data_ptr())
    try:
        scn.set_math_mode(math)
        for ch in (32, 64):
            rs = np.random.RandomState(ch)
            x = rs.randn(n, ch).astype(np.float32)
            w = (rs.randn(27, 1, ch, ch) * (2.0 / (ch * 27)) ** 0.5).astype(np.float32)
            want, _ = so.o_conv_forward(x, w, rules, n)
            xt, wt = T(x), T(w)
            out = torch.empty(n, ch, device="cuda")
            stats = _stats_buffer()
            macs = C.c_double()
            check(lib().scn_fuse_next_stats(p(stats)))
            check(lib().scn_submanifold_convolution_forward(G.m._h, l3(full), l3([3, 3, 3]), p(xt), p(out), p(wt), None, ch, ch, C.byref(macs), None, 0, None, None))
            took_l, took_s = C.c_int(), C.c_int()
            check(lib().scn_fuse_result(C.byref(took_l), C.byref(took_s)))
            torch.cuda.synchronize()
            assert took_s.value == 1 and took_l.value == 0
            _close(out.cpu().numpy(), want, *TC_TOL[math])
            s1, s2 = _reduce_stats(stats, ch)
            o64 = out.double()
            np.testing.assert_allclose(s1, o64.sum(0).cpu().numpy(), rtol=1e-4, atol=1e-3 * n ** 0.5)
            np.testing.assert_allclose(s2, (o64 * o64).sum(0).cpu().numpy(), rtol=1e-4)
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ odd channel counts: padded copy + bf16 copy in one launch
@pytest.mark.parametrize("math", ["tf32", "bf16"])
def test_odd_channel_counts_use_separate_scratch(math):
    """Cin = 48 with Cout = 256 (no packing) and a Deconvolution with Cin = 48: the rows are zero-padded to 64 channels into
    one scratch buffer and, in bf16 mode, converted into a SECOND one (round 1 used the same buffer for both)."""
    scn = _scn()
    _tc_or_skip(scn)
    c = synthetic.small_building(40, 36, 12, 3, seed=4)
    full, coarse = [64, 64, 32], [32, 32, 16]
    G, O = _gpu(), so.OracleMetadata()
    n = G.input_layer(full, c, 0, 4)
    O.input_layer(full, c, 0, 4)
    rules2 = O.conv_rules(full, coarse, [2, 2, 2], [2, 2, 2])
    nc = O.nactive(coarse)
    rs = np.random.RandomState(48)
    x = rs.randn(n, 48).astype(np.float32)
    w = (rs.randn(27, 1, 48, 256) * (2.0 / (48 * 27)) ** 0.5).astype(np.float32)
    want, _ = so.o_conv_forward(x, w, O.submanifold_rules(full, [3, 3, 3]), n)
    xc = rs.randn(nc, 48).astype(np.float32)
    wd = (rs.randn(8, 1, 48, 64) * (2.0 / (48 * 8)) ** 0.5).astype(np.float32)
    wantd, _ = so.o_conv_forward(xc, wd, rules2, n, deconv=True)
    dy = rs.randn(n, 256).astype(np.float32)
    din_w, dw_w = so.o_conv_backward(x, dy, w, O.submanifold_rules(full, [3, 3, 3]))
    try:
        scn.set_math_mode(math)
        out, outd = torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([3, 3, 3]), G.m, T(x), out, T(w), torch.Tensor())
        scn.SCN.Convolution_updateOutput(L(full), L(coarse), L([2, 2, 2]), L([2, 2, 2]), G.m, T(rs.randn(n, 48).astype(np.float32)), torch.empty(0, device="cuda"),
                                         T((rs.randn(8, 1, 48, 64) * 0.05).astype(np.float32)), torch.Tensor())
        scn.SCN.Deconvolution_updateOutput(L(coarse), L(full), L([2, 2, 2]), L([2, 2, 2]), G.m, T(xc), outd, T(wd), torch.Tensor())
        din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
        scn.SCN.SubmanifoldConvolution_backward(L(full), L([3, 3, 3]), G.m, T(x), din, T(dy), T(w), dw, torch.Tensor())
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    rtol, atol = TC_TOL[math]
    _close(out.cpu().numpy(), want, rtol, atol)
    _close(outd.cpu().numpy(), wantd, rtol, atol)
    _close(din.cpu().numpy(), din_w, rtol, atol)
    _close(dw.cpu().numpy(), dw_w, rtol, atol)


# ------------------------------------------------------------------ the benchmarked path vs the reference's outputs
@pytest.mark.parametrize("math", ["bf16", "tf32"])
def test_replayed_program_tensor_core_vs_reference_golden(math):
    """What bench.py times: tensor-core math mode + REPLAYED program on an internally numbered Metadata, on the sw4c backbone
    (128-channel <1,4,1> kernel, level 0 with >= 32768 rows => bf16-only outputs in bf16 mode) against the outputs of the
    reference's own scn.FPN_Net (tests/golden/fpn_sw4c_mid.npz).  Replayed twice.  Counters prove the lateral stage, the
    epilogue statistics and the bf16-only outputs were taken and that no lateral fell back to a separate pass."""
    scn = _scn()
    _tc_or_skip(scn)
    cfg = scn.sw4c_fpn432_config()
    bld = dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)
    g = np.load(os.path.join(GOLD, "fpn_sw4c_mid.npz"))
    try:
        scn.set_math_mode(math)
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().eval()
        coords = synthetic.building_coords(**bld)
        c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()
        with torch.no_grad():
            net([c, f])  # records (layer by layer)
            assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
            for rep in range(2):
                before = _counters()
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])  # replays
                torch.cuda.synchronize()
                d = _delta(before)
                assert scn.forward_pass_multiplyAdd_count == float(g["macs"])
                # 8 top-down steps: deconvolution + lateral shortcut in one launch each; none may fall back
                assert d["lateral"] == 8 and d["lateral_fallback"] == 0, d
                assert d["stats"] >= 8 and d["bn_from_sums"] >= 8, d
                assert d["simt"] == 0, d
                if math == "bf16":
                    assert d["half_only"] >= 3, d
                worst = 0.0
                for tag, maps in (("rpn", rpn), ("roi", roi)):
                    assert len(maps) == int(g[f"n_{tag}"])
                    for i, m in enumerate(maps):
                        assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
                        ref = g[f"{tag}{i}_features"]
                        err = float(np.abs(m.features.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max()))
                        worst = max(worst, err)
                        assert err < TC_E2E[math], (tag, i, err, rep)
                print(f"[pin] {math} replay {rep}: worst map error {worst:.3e} of max|ref| (tolerance {TC_E2E[math]})", d)
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ whole-network training step vs the reference's autograd
@pytest.mark.parametrize("math", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("replay", [False, True])
def test_whole_network_training_step_vs_reference_autograd(math, replay):
    """replay=True: the SECOND training step of the network, i.e. the recorded program replayed in training mode (one autograd node,
    scn_program_run + scn_program_backward) from the same initial state.  Train-mode forward (batch statistics, running statistics updated), loss = sum of mean(f^2) over the returned maps,
    autograd backward through every layer kind, against the same step of the reference's scn.FPN_Net on its CPU extension
    (tests/golden/fpn_mini4_train.npz, tests/golden/make_golden.py::run_reference_fpn_train).  Parameters of the dead
    top-down levels get no gradient on either side.  Tolerances per parameter tensor (worst element / max|grad|, relative
    rms) and on the cosine of the whole gradient vector: stated next to the measured values below."""
    scn = _scn()
    if math != "fp32":
        _tc_or_skip(scn)
    g = np.load(os.path.join(GOLD, "fpn_mini4_train.npz"))
    cfg = dict(fpn_util.mini4_config(), track_running_stats=True)
    bld = dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)
    # gradients pass through ~40 operand-rounded layers forward AND backward: the bound is on the whole tensor (relative rms)
    # and, looser, on its worst element
    # Measured on B200 (tools/grad_error.py, gpurun_out/r2_grad_error.log): fp32 <= 7e-6 everywhere; tf32 rel rms <= 4.8e-2, worst element
    # 1.4e-1; bf16 rel rms <= 1.35e-1, worst element 3.6e-1 (train-mode BatchNorm over the few dozen rows of the deepest level
    # amplifies operand rounding; the errors scale with the operand precision, tf32 : bf16 ~ 1 : 2.5, in every tensor).
    tol_max, tol_rms, tol_cos = {"fp32": (5e-3, 5e-3, 0.99999), "tf32": (2.5e-1, 8e-2, 0.995), "bf16": (5e-1, 2e-1, 0.98)}[math]
    tol = {"fp32": 5e-3, "tf32": 3e-2, "bf16": 8e-2}[math]
    try:
        scn.set_math_mode(math)
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().train()
        coords = synthetic.building_coords(**bld)
        if replay:  # first step records; then back to the initial state (in place: the program keeps the parameter tensors)
            rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
            sum((m.features ** 2).mean() for m in rpn + roi).backward()
            assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
            net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
            net.zero_grad(set_to_none=True)
            n0 = scn.SCN.lib().scn_debug_counter(11)
        rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
        maps = rpn + roi
        assert len(maps) == int(g["n_maps"])
        terms = [(m.features ** 2).mean() for m in maps]
        loss = sum(terms)
        loss.backward()
        torch.cuda.synchronize()
        if replay:
            assert scn.SCN.lib().scn_debug_counter(11) == n0 + 1, "the backward pass did not run through scn_program_backward"
    finally:
        scn.set_math_mode("fp32")
    np.testing.assert_allclose(np.array([float(t) for t in terms]), g["map_mean_sq"], rtol=tol)
    assert abs(float(loss) - float(g["loss"])) <= tol * float(g["loss"])
    want_keys = {k[5:] for k in g.files if k.startswith("grad:")}
    got = {k: p.grad for k, p in net.named_parameters()}
    assert {k for k, v in got.items() if v is not None} == want_keys
    worst, table = ("", 0.0), []
    for k in want_keys:
        ref = g["grad:" + k].astype(np.float64)
        d = got[k].cpu().numpy().astype(np.float64) - ref
        err = float(np.abs(d).max() / max(1e-6, np.abs(ref).max()))
        rms = float(np.sqrt((d * d).mean()) / max(1e-12, np.sqrt((ref * ref).mean())))
        table.append((err, rms, k))
        if err > worst[1]:
            worst = (k, err)
    table.sort(reverse=True)
    print("[pin] training step %s, per-parameter gradient error (max / max|ref|, rel rms):" % math)
    for err, rms, k in table[:12]:
        print("        %-40s %.3e %.3e" % (k, err, rms))
    for err, rms, k in table:
        assert err < tol_max and rms < tol_rms, (k, err, rms)
    keys = sorted(want_keys)
    a = np.concatenate([got[k].cpu().numpy().ravel() for k in keys]).astype(np.float64)
    b = np.concatenate([g["grad:" + k].ravel() for k in keys]).astype(np.float64)
    cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)))
    print(f"[pin] training step {math}: cosine of the whole gradient vector with the reference's {cos:.6f}")
    assert cos >= tol_cos, cos
    for k, b in net.named_buffers():
        ref = g["buf:" + k]
        np.testing.assert_allclose(b.cpu().numpy(), ref, rtol=tol, atol=tol * max(1e-3, float(np.abs(ref).max())), err_msg=k)
    print(f"[pin] training step {math}: worst gradient error {worst[1]:.3e} of max|grad| ({worst[0]})")


# ------------------------------------------------------------------ next rows (SURVEY.md section 8f): RPN head + anchors, SparseToDense
def test_rpn_head_and_anchors_vs_reference_golden():
    """detection_3d_b200.rpn.RPNHead / AnchorGenerator (one CUDA kernel per map each) against the outputs of the reference's own
    RPNHead.forward / AnchorGenerator.grid_anchors (tests/golden/rpn_sw4c_mid.npz) and against the CPU oracle on ragged sizes."""
    from detection_3d_b200 import rpn
    from oracle import rpn_oracle as ro
    g = np.load(os.path.join(GOLD, "rpn_sw4c_mid.npz"))
    f = np.load(os.path.join(GOLD, "fpn_sw4c_mid.npz"))
    head = rpn.RPNHead(128, 4, 2)
    head.load_state_dict({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")})
    head = head.cuda().eval()
    gen = rpn.sw4c_anchor_generator()
    n = int(g["n_maps"])
    feats = [T(f[f"rpn{i}_features"]) for i in range(n)]
    with torch.no_grad():
        logits, regs = head([x.t().unsqueeze(0).unsqueeze(3) for x in feats])  # the reference's [1, C, n, 1] layout
        logits2, _ = head(feats)                                               # plain rows
        anchors = gen.grid_anchors([torch.from_numpy(f[f"rpn{i}_locations"].astype(np.int64)) for i in range(n)])
    torch.cuda.synchronize()
    for i in range(n):
        assert tuple(logits[i].shape) == g[f"logits{i}"].shape and tuple(regs[i].shape) == g[f"reg{i}"].shape
        np.testing.assert_allclose(logits[i].cpu().numpy(), g[f"logits{i}"], rtol=1e-4, atol=1e-6)  # fp32, summation order only
        np.testing.assert_allclose(regs[i].cpu().numpy(), g[f"reg{i}"], rtol=1e-4, atol=1e-6)
        assert torch.equal(logits[i], logits2[i])
        assert np.array_equal(anchors[i].cpu().numpy(), g[f"anchors{i}"])  # bit exact
    # ragged / edge shapes against the oracle: 1 row, a non-multiple of the row tile, 0 rows, other channel counts and group counts
    rs = np.random.RandomState(5)
    for rows, c, A, sep in [(1, 128, 4, 2), (13, 64, 2, 1), (0, 128, 4, 2), (777, 256, 3, 3)]:
        h = rpn.RPNHead(c, A, sep).cuda()
        with torch.no_grad():
            for p_ in h.parameters():
                p_.copy_(torch.from_numpy((rs.randn(*p_.shape) * 0.1).astype(np.float32)))
        x = rs.randn(rows, c).astype(np.float32)
        with torch.no_grad():
            lg, rg = h([T(x)])
        if rows == 0:  # (torch's conv2d -- what the reference runs -- rejects an empty map; ours returns empty outputs)
            assert tuple(lg[0].shape) == (1, 0, A, sep) and tuple(rg[0].shape) == (1, 0, A, 7 * sep)
            continue
        sd = {k: v.detach().cpu().numpy() for k, v in h.state_dict().items()}
        wl, wr = ro.rpn_head_forward(x, sd["conv.weight"], sd["conv.bias"], sd["cls_logits.weight"], sd["cls_logits.bias"], sd["bbox_pred.weight"],
                                     sd["bbox_pred.bias"], A, sep)
        assert tuple(lg[0].shape) == wl.shape and tuple(rg[0].shape) == wr.shape
        if rows:
            _close(lg[0].cpu().numpy(), wl, 1e-4, 1e-5)
            _close(rg[0].cpu().numpy(), wr, 1e-4, 1e-5)


def test_rpn_on_backbone_outputs_end_to_end():
    """BASELINE.json config 3 up to the proposals' inputs: backbone (fp32 mode) -> RPN head + anchors on its four rpn maps with
    device-resident locations, against the reference's outputs for the same building (golden): same rows, same order."""
    scn = _scn()
    from detection_3d_b200 import rpn
    g = np.load(os.path.join(GOLD, "rpn_sw4c_mid.npz"))
    cfg = scn.sw4c_fpn432_config()
    try:
        scn.set_math_mode("fp32")
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().eval()
        head = rpn.RPNHead(128, 4, 2)
        head.load_state_dict({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")})
        head = head.cuda().eval()
        gen = rpn.sw4c_anchor_generator()
        coords = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
        with torch.no_grad():
            rpn_maps, _ = net([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
            logits, regs = head([m.features for m in rpn_maps])
            anchors, scopes = gen(None, rpn_maps)
            obj, reg = rpn.cat_scales_obj_reg(logits, regs, scopes)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    for i in range(4):
        assert np.array_equal(anchors[i].cpu().numpy(), g[f"anchors{i}"])
        _close(logits[i].cpu().numpy(), g[f"logits{i}"], 2e-3, 2e-4)  # backbone fp32 end-to-end tolerance carried through the head
        _close(regs[i].cpu().numpy(), g[f"reg{i}"], 2e-3, 2e-4)
    n_anchor = sum(a.shape[0] for a in anchors)
    assert tuple(obj.shape) == (n_anchor, 2) and tuple(reg.shape) == (n_anchor, 14)
    assert torch.equal(obj[:anchors[0].shape[0]], logits[0].reshape(-1, 2))


@pytest.mark.parametrize("case", ["golden", "building", "big"])
def test_sparse_to_dense_forward_backward(case):
    """scn.SparseToDense (+ rulebook kind 3, bit exact) against the reference package's outputs (golden, two batch items) and the
    CPU oracle; `big` = the level-4 roi map size of the B470 building ([128, 128, 32] x 128 planes)."""
    scn = _scn()
    g = np.load(os.path.join(GOLD, "sparse_to_dense.npz"))
    rs = np.random.RandomState(3)
    if case == "golden":
        coords, feats, sz = g["coords"], g["feats"], [16, 16, 8]
    elif case == "building":
        coords = np.concatenate([synthetic.small_building(40, 36, 12, 3, seed=4), synthetic.small_building(30, 30, 10, 2, seed=5, batch_index=1)])
        feats, sz = rs.randn(coords.shape[0], 20).astype(np.float32), [64, 64, 32]
    else:
        c0 = synthetic.building_coords()
        coords = np.unique(np.concatenate([c0[:, :3] >> 4, c0[:, 3:]], 1), axis=0)
        feats, sz = rs.randn(coords.shape[0], 128).astype(np.float32), [128, 128, 32]
    inp = scn.InputLayer(3, sz, mode=4)
    ft = T(feats).requires_grad_(True)
    x = inp([torch.from_numpy(coords.astype(np.int64)), ft])
    dense = scn.SparseToDense(3, feats.shape[1])(x)
    O = so.OracleMetadata()
    n = O.input_layer(sz, coords, 0, 4)
    rules = O.sparse_to_dense_rules(sz)
    got_rules = [t.numpy() for t in x.metadata.sparseToDenseRuleBook(sz)]
    assert len(got_rules) == len(rules)
    for a, b in zip(got_rules, rules):
        assert np.array_equal(a, b)
    want = so.o_sparse_to_dense_forward(x.features.detach().cpu().numpy(), rules, sz)
    assert tuple(dense.shape) == want.shape
    assert np.array_equal(dense.detach().cpu().numpy(), want)
    w = rs.randn(*want.shape).astype(np.float32)
    (dense * T(w)).sum().backward()
    hdr, tab = O.input_rules()
    want_g = so.o_input_layer_backward(so.o_sparse_to_dense_backward(w, rules, n), hdr, tab)
    np.testing.assert_allclose(ft.grad.cpu().numpy(), want_g, rtol=1e-6, atol=1e-7)
    crop = scn.sparse_3d_to_dense_2d(x)
    ext = (coords[:, :3].max(0) + 1).tolist()
    assert tuple(crop.shape[2:]) == tuple(ext)
    if case == "golden":
        # (the voxel means of the input layer differ from the CPU's in the last bit: fused multiply-add; the scatter itself is exact, above)
        np.testing.assert_allclose(dense.detach().cpu().numpy(), g["dense"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(crop.detach().cpu().numpy(), g["crop"], rtol=1e-6, atol=1e-7)
        dense2 = scn.SparseToDense(3, 6)(x)
        (dense2 * T(g["w"])).sum().backward()  # (second backward accumulates: compare the increment)
        np.testing.assert_allclose(ft.grad.cpu().numpy() - want_g, g["grad_feats"], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ ROIAlignRotated3D (SURVEY.md section 8f rank 3)
def _roi_case(rs, ext, n_rois, batch):
    cw, ch, cz = rs.uniform(-1, ext[1] + 1, n_rois), rs.uniform(-1, ext[0] + 1, n_rois), rs.uniform(-0.5, ext[2] + 0.5, n_rois)
    w, h, z = rs.uniform(0.3, 9, n_rois), rs.uniform(0.3, 9, n_rois), rs.uniform(0.3, 6, n_rois)
    th = rs.uniform(-180, 180, n_rois)
    th[:3] = [0, 90, -45]
    b = rs.randint(0, batch, n_rois)
    return np.stack([b, cw, ch, cz, w, h, z, th], 1).astype(np.float32)


def _roi_inputs(case, sampling):
    """The seeded inputs of one ROIAlignRotated3D case (also read by tests/golden/make_golden_roialign.py): coordinates, features,
    map size, channels, pooled size, spatial scale, cropped extent, batch size, rois and the gradient of the output."""
    rs = np.random.RandomState(17 + sampling)
    if case == "small2":
        coords = np.concatenate([synthetic.small_building(20, 18, 8, 2, seed=4), synthetic.small_building(16, 22, 6, 2, seed=5, batch_index=1)])
        sz, C_, n_rois, pooled, scale = [32, 32, 8], 12, 40, (3, 4, 2), 0.5
    else:
        c0 = synthetic.building_coords()
        coords = np.unique(np.concatenate([c0[:, :3] >> 4, c0[:, 3:]], 1), axis=0)
        sz, C_, n_rois, pooled, scale = [128, 128, 32], 128, 24, (7, 7, 7), 0.25
    feats = rs.randn(coords.shape[0], C_).astype(np.float32)
    ext = (coords[:, :3].max(0) + 1).tolist()
    batch = int(coords[:, 3].max()) + 1
    rois = _roi_case(rs, [e / scale for e in ext], n_rois, batch)  # roi coordinates are in input units: the kernel multiplies by spatial_scale
    g = rs.randn(n_rois, C_, *pooled).astype(np.float32)
    return coords, feats, sz, C_, pooled, scale, ext, batch, rois, g


def _close_golden(got, gold, key, rtol, atol):
    """_close on the entries of `got` stored under `key` of the golden file, scaled by the max|.| of the whole stored array."""
    got = np.asarray(got)
    assert got.shape == tuple(gold[key + "_shape"])
    scale = max(1.0, float(gold[key + "_absmax"]))
    np.testing.assert_allclose(got.ravel()[gold[key + "_idx"]], gold[key], rtol=rtol, atol=atol * scale)
    np.testing.assert_allclose(np.abs(got).max(), gold[key + "_absmax"], rtol=rtol, atol=atol * scale)


def _roi_align_vs_restatement(case, sampling):
    """detection_3d_b200.roi_align.ROIAlignRotated3D (samples the SPARSE map) against the CPU restatement (oracle) of the reference's
    kernels on the densified, cropped map -- exactly the reference module's data flow.  Forward and backward (down to the input
    features).  Returns what the reference comparison needs: output, restated output, restated map gradient, dense map, inputs."""
    scn = _scn()
    from detection_3d_b200.roi_align import ROIAlignRotated3D
    coords, feats, sz, C_, pooled, scale, ext, batch, rois, g = _roi_inputs(case, sampling)
    inp = scn.InputLayer(3, sz, mode=4)
    ft = T(feats).requires_grad_(True)
    x = inp([torch.from_numpy(coords.astype(np.int64)), ft])
    layer = ROIAlignRotated3D(pooled, scale, sampling)
    out = layer(x, T(rois))
    assert tuple(out.shape) == g.shape
    out.backward(T(g))
    torch.cuda.synchronize()
    dense = scn.sparse_3d_to_dense_2d(x).detach().contiguous()          # what the reference module samples
    assert list(dense.shape[2:]) == ext
    want = so.o_roi_align_rotated_3d_forward(dense.cpu().numpy(), rois, scale, pooled, sampling)
    _close(out.detach().cpu().numpy(), want, 1e-5, 2e-5)
    dd = so.o_roi_align_rotated_3d_backward(g, rois, scale, pooled, sampling, tuple(dense.shape))
    full = np.zeros((batch, C_) + tuple(sz), np.float32)
    full[:, :, :ext[0], :ext[1], :ext[2]] = dd
    O = so.OracleMetadata()
    n = O.input_layer(sz, coords, 0, 4)
    hdr, tab = O.input_rules()
    want_g = so.o_input_layer_backward(so.o_sparse_to_dense_backward(full, O.sparse_to_dense_rules(sz), n), hdr, tab)
    _close(ft.grad.cpu().numpy(), want_g, 1e-4, 5e-5)
    return out, want, dd, dense, (C_, pooled, scale, ext, batch, rois, g)


@pytest.mark.parametrize("case", ["small2", "level4"])
@pytest.mark.parametrize("sampling", [2, 0])
def test_roi_align_rotated_3d_vs_restatement_and_golden(case, sampling):
    """ROIAlignRotated3D against the CPU restatement (_roi_align_vs_restatement), and both against tests/golden/roi_align_rotated_3d.npz:
    a regression pin of the restatement's outputs for these inputs (a seeded sample of every output, tests/golden/
    make_golden_roialign.py), so that the product and the restatement cannot drift together.  Rois inside, straddling and outside the
    map, degenerate sizes, sampling ratio 2 and adaptive.  Tolerance 2e-5 of max|ref|: fp32, the order of the 8-corner sum and FMA
    contraction differ."""
    out, want, dd, _, _ = _roi_align_vs_restatement(case, sampling)
    gold = np.load(os.path.join(GOLD, "roi_align_rotated_3d.npz"))
    key = f"{case}_s{sampling}"
    _close_golden(out.detach().cpu().numpy(), gold, key + "_fwd", 1e-5, 2e-5)
    _close_golden(want, gold, key + "_fwd", 1e-5, 2e-5)
    _close_golden(dd, gold, key + "_bwd", 1e-4, 5e-5)


@pytest.mark.skipif(not os.path.exists(os.path.join(os.path.dirname(so.__file__), "_ref", "libroialign3d_ref.so")),
                    reason="needs the reference's ROIAlignRotated3D kernels built into oracle/_ref (make -C oracle ref, from the reference's sources)")
@pytest.mark.parametrize("case", ["small2", "level4"])
@pytest.mark.parametrize("sampling", [2, 0])
def test_roi_align_rotated_3d_vs_reference_kernel(case, sampling):
    """ROIAlignRotated3D and the CPU restatement against the reference's own CUDA kernels compiled unmodified
    (oracle/_ref/libroialign3d_ref.so) on the densified, cropped map.  Same cases and tolerances as above."""
    out, want, dd, dense, (C_, pooled, scale, ext, batch, rois, g) = _roi_align_vs_restatement(case, sampling)
    ref = so.roi_align_ref_lib()
    p = lambda t: C.c_void_p(t.data_ptr())
    n_rois = rois.shape[0]
    r_t = T(rois)
    out_ref = torch.empty_like(out)
    assert ref.ref_roi_align_rotated_3d_forward(p(dense), batch, C_, ext[0], ext[1], ext[2], p(r_t), n_rois, scale, pooled[0], pooled[1], pooled[2], sampling, p(out_ref)) == 0
    _close(out.detach().cpu().numpy(), out_ref.cpu().numpy(), 1e-5, 2e-5)
    _close(want, out_ref.cpu().numpy(), 1e-5, 2e-5)                      # pins the CPU restatement too
    d_ref = torch.empty_like(dense)
    g_t = T(g)
    assert ref.ref_roi_align_rotated_3d_backward(p(g_t), p(r_t), n_rois, scale, pooled[0], pooled[1], pooled[2], batch, C_, ext[0], ext[1], ext[2], sampling, p(d_ref)) == 0
    _close(dd, d_ref.cpu().numpy(), 1e-4, 5e-5)


# ------------------------------------------------------------------ RPN post-processing and voxeliser (SURVEY.md section 8f rank 4)
def _rpn_golden_inputs():
    r = np.load(os.path.join(GOLD, "rpn_sw4c_mid.npz"))
    nm = int(r["n_maps"])
    anchors = np.concatenate([r[f"anchors{i}"] for i in range(nm)], 0)
    logits = np.concatenate([r[f"logits{i}"].reshape(-1, r[f"logits{i}"].shape[-1]) for i in range(nm)], 0)
    regs = np.concatenate([r[f"reg{i}"].reshape(-1, r[f"reg{i}"].shape[-1]) for i in range(nm)], 0)
    return anchors, logits, regs


def test_box_decode_and_top_k_vs_reference_golden():
    """BoxCoder3D.decode (one class, two classes per anchor, weights) against the reference's own decode; top_k against torch.topk."""
    from detection_3d_b200 import postproc as pp
    g = np.load(os.path.join(GOLD, "postproc.npz"))
    OS, RS = np.float32(g["obj_scale"]), np.float32(g["reg_scale"])
    anchors, logits, regs = _rpn_golden_inputs()
    coder = pp.BoxCoder3D()
    _close(coder.decode(T(regs[:, :7] * RS), T(anchors)).cpu().numpy(), g["decode_1"], 2e-6, 2e-6)
    _close(coder.decode(T(regs[:500] * RS), T(anchors[:500])).cpu().numpy(), g["decode_2"], 2e-6, 2e-6)
    _close(pp.BoxCoder3D(weights=(10., 10., 5., 5., 5., 5., 2.)).decode(T(regs[:500, :7] * RS), T(anchors[:500])).cpu().numpy(), g["decode_w"], 2e-6, 2e-6)
    idx = torch.randperm(anchors.shape[0], generator=torch.Generator().manual_seed(0))[:777].cuda()
    assert torch.equal(coder.decode(T(regs[:, :7] * RS), T(anchors), indices=idx), coder.decode(T(regs[:, :7] * RS), T(anchors))[idx])
    v = T(logits[:, 0] * OS)
    for k, sig in ((1500, True), (v.numel(), False), (1, True), (0, False)):
        got_v, got_i = pp.top_k(v, k, sigmoid=sig)
        ref_v, ref_i = torch.topk(v.sigmoid() if sig else v, k, sorted=True)
        assert torch.equal(got_v, ref_v)
        assert torch.equal((v.sigmoid() if sig else v)[got_i], ref_v)  # (indices of equal values may legitimately differ)
    ties = torch.tensor([0.5, 2.0, 0.5, 2.0, -1.0, 2.0], device="cuda")
    tv, ti = pp.top_k(ties, 5)
    assert ti.tolist() == [1, 3, 5, 0, 2] and tv.tolist() == [2.0, 2.0, 2.0, 0.5, 0.5]  # ties: lower index first
    big = torch.randn(200000, generator=torch.Generator().manual_seed(1)).cuda()
    bv, bi = pp.top_k(big, 3000)
    assert torch.equal(bv, torch.topk(big, 3000)[0]) and torch.equal(big[bi], bv)


def test_boxes_iou_3d_vs_reference_golden_and_oracle():
    """Rotated BEV IoU (all criteria) and 3-D IoU against the reference's numba kernel outputs (golden) and the CPU restatement on
    random + degenerate boxes.  Tolerance 3e-5 absolute: float32 polygon clipping vs the reference's vertex sort + triangle fan."""
    from detection_3d_b200 import postproc as pp
    from oracle import postproc_oracle as po
    g = np.load(os.path.join(GOLD, "postproc.npz"))
    b5, rows, qs = g["iou2d_boxes"], g["iou2d_rows"], g["iou2d_query_sel"]
    to7 = lambda b: np.stack([b[:, 0], b[:, 1], np.zeros(len(b)), b[:, 2], b[:, 3], np.ones(len(b)), b[:, 4]], 1).astype(np.float32)
    for crit in (-1, 0, 1, 2, 3):
        got = pp.boxes_iou_3d(T(to7(b5[rows])), T(to7(b5[qs])), None, criterion=crit, only_xy=True, flag='rpn_post').cpu().numpy()
        np.testing.assert_allclose(got, g[f"iou2d_c{crit}"], rtol=2e-4, atol=3e-5)
    t7, a7 = g["iou3d_targets"], g["iou3d_anchors"]
    np.testing.assert_allclose(pp.boxes_iou_3d(T(t7), T(a7), None, flag='rpn_post').cpu().numpy(), g["iou3d_plain"], rtol=2e-4, atol=3e-5)
    aug = {'target_Y': 0.3, 'target_Z': 0.4, 'anchor_Y': 0.0, 'anchor_Z': 0.0}
    np.testing.assert_allclose(pp.boxes_iou_3d(T(t7), T(a7), aug, criterion=1, flag='rpn_label_generation').cpu().numpy(), g["iou3d_aug"], rtol=2e-4, atol=3e-5)
    np.testing.assert_allclose(pp.boxes_iou_3d(T(t7), T(a7), None, only_xy=True, flag='roi_post').cpu().numpy(), g["iou3d_xy"], rtol=2e-4, atol=3e-5)
    with pytest.raises(AssertionError):
        pp.boxes_iou_3d(T(t7), T(a7), aug, flag='rpn_post')  # the reference asserts aug_thickness is None here
    rs = np.random.RandomState(5)
    n = 40
    b = np.stack([rs.uniform(0, 5, n), rs.uniform(0, 5, n), rs.uniform(0, 2, n), rs.uniform(0.1, 3, n), rs.uniform(0.1, 3, n), rs.uniform(0.1, 2, n), rs.uniform(-4, 4, n)], 1).astype(np.float32)
    b[1] = b[0]                      # identical
    b[2, 3] = 0.01                   # a very thin box
    b[3] = [1, 1, 0, 2, 2, 1, 0]; b[4] = [1, 1, 0.5, 2, 2, 1, 0]; b[5] = [3, 1, 0, 2, 2, 1, 0]  # same square, shifted in z; touching square
    got = pp.boxes_iou_3d(T(b), T(b), None, flag='rpn_post').cpu().numpy()
    want = po.boxes_iou_3d(b, b)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    np.testing.assert_allclose(np.nan_to_num(got), np.nan_to_num(want), rtol=2e-4, atol=3e-5)
    assert got[0, 1] == pytest.approx(1.0, abs=1e-6) and got[3, 5] == 0.0
    assert pp.boxes_iou_3d(T(b[:0]), T(b), None, flag='rpn_post').shape == (0, n)


def test_rotate_nms_3d_and_rpn_post_processor_vs_reference_golden():
    """The whole chain of inference_3d.py:82-161 for one example against the reference's own RPNPostProcessor output (bit-exact
    selection and order of the surviving boxes; box values to 2e-6), rotate_nms_3d on its own, and -- at the B470 size (9,248
    anchors -> 1,500 candidates) -- against the CPU restatement."""
    from detection_3d_b200 import postproc as pp
    from oracle import postproc_oracle as po
    g = np.load(os.path.join(GOLD, "postproc.npz"))
    OS, RS = np.float32(g["obj_scale"]), np.float32(g["reg_scale"])
    anchors, logits, regs = _rpn_golden_inputs()
    sel = g["rpn_sel"]
    anc, obj, reg = anchors[sel], logits[sel, 0] * OS, regs[sel, :7] * RS
    post = pp.RPNPostProcessor(batch_size=1, fpn_pre_nms_top_n=130, fpn_post_nms_top_n=105, nms_thresh=0.1, nms_aug_thickness=[0.3, 0.3], min_size=0).eval()
    res = post(pp.Boxes3D(T(anc)), T(obj), T(reg))
    assert len(res) == 1 and tuple(res[0].bbox3d.shape) == g["rpn_boxes"].shape
    _close(res[0].bbox3d.cpu().numpy(), g["rpn_boxes"], 2e-6, 2e-6)
    np.testing.assert_allclose(res[0].get_field("objectness").cpu().numpy(), g["rpn_objectness"], rtol=2e-6, atol=1e-7)
    dec = pp.BoxCoder3D().decode(T(reg), T(anc))
    keep = pp.rotate_nms_3d(dec[:150], T(obj[:150]), pre_max_size=120, post_max_size=60, iou_threshold=0.3, flag='rpn_post')
    assert np.array_equal(keep.cpu().numpy(), g["nms_keep_03"])
    assert pp.rotate_nms_3d(dec[:0], T(obj[:0]), 100, 50, 0.3).numel() == 0
    # two examples in one batch = the two halves processed independently
    half = anc.shape[0] // 2
    both = pp.Boxes3D(T(anc), examples_idxscope=torch.tensor([[0, half], [half, anc.shape[0]]]))
    r2 = post(both, T(obj), T(reg))
    one = post(pp.Boxes3D(T(anc[half:])), T(obj[half:]), T(reg[half:]))
    assert len(r2) == 2 and torch.equal(r2[1].bbox3d, one[0].bbox3d)
    # every anchor of the four rpn maps against the CPU restatement (260 candidates: the pure-Python oracle needs ~40 us per pair)
    full_obj, full_reg = logits[:, 0] * OS, regs[:, :7] * RS
    mid = pp.RPNPostProcessor(1, 260, 150, 0.1, [0.3, 0.3], 0).eval()
    got = mid(pp.Boxes3D(T(anchors)), T(full_obj), T(full_reg))[0]
    wb, wo = po.rpn_post_process(anchors, full_obj, full_reg, 260, 150, 0.1, (0.3, 0.3))
    assert tuple(got.bbox3d.shape) == wb.shape
    _close(got.bbox3d.cpu().numpy(), wb, 2e-6, 2e-6)
    np.testing.assert_allclose(got.get_field("objectness").cpu().numpy(), wo, rtol=2e-6, atol=1e-7)
    # full size of the B470 configuration (sw4c's top-n, tools/train_net_sparse3d.py:247-255: 1,500 candidates -> 2.25 M pairs), checked
    # through the property that DEFINES greedy suppression: with S[i, j] = (3-D IoU > 0 and BEV IoU >= thresh) over the candidates in
    # score order, no kept box is suppressed by an earlier kept box, and every dropped box is suppressed by an earlier kept box.
    cand_obj, cand_idx = pp.top_k(T(full_obj), 1500, sigmoid=True)
    cand = pp.BoxCoder3D().decode(T(full_reg), T(anchors), indices=cand_idx)
    aug = cand.clone()
    aug[:, 3:5] = torch.clamp(aug[:, 3:5], min=0.3)
    aug[:, 5] = torch.clamp(aug[:, 5], min=0.3)
    keep = pp.rotate_nms_3d(aug, cand_obj, pre_max_size=2000, post_max_size=1500, iou_threshold=0.1, flag='rpn_post')
    S = (pp.boxes_iou_3d(aug, aug, None, flag='rpn_post') > 0) & (pp.boxes_iou_3d(aug, aug, None, only_xy=True, flag='rpn_post') >= 0.1)
    S = torch.triu(S, diagonal=1)
    kept = torch.zeros(1500, dtype=torch.bool, device="cuda")
    kept[keep] = True
    assert torch.equal(keep, torch.sort(keep)[0]) and 0 < keep.numel() < 1500
    by_kept = S[kept].any(0)                       # suppressed by some earlier kept box
    assert not (by_kept & kept).any() and (by_kept | kept).all()
    big = pp.RPNPostProcessor(1, 1500, 750, 0.1, [0.3, 0.3], 0).eval()(pp.Boxes3D(T(anchors)), T(full_obj), T(full_reg))[0]
    n_out = min(750, keep.numel())
    assert torch.equal(big.bbox3d, cand[keep[:n_out]]) and torch.equal(big.get_field("objectness"), cand_obj[keep[:n_out]])


def test_voxelize_vs_reference_golden():
    """Input voxeliser against the statements of the reference's SUNCGDataset.__getitem__ executed on the same points (golden): integer
    voxel coordinates bit-exact, features to float32 rounding, dropped rows identical; B470-sized cloud against the CPU restatement."""
    from detection_3d_b200 import postproc as pp
    from oracle import postproc_oracle as po
    g = np.load(os.path.join(GOLD, "postproc.npz"))
    pcl = g["vox_pcl"]
    locs, feats, size3d = pp.voxelize(T(pcl[:, :3].copy()), T(pcl), 50, [2048, 2048, 512])
    assert np.array_equal(locs.cpu().numpy(), g["vox_locs"])
    np.testing.assert_allclose(feats.cpu().numpy(), g["vox_feats"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(size3d.numpy(), g["vox_size3d"], rtol=1e-6)
    locs, feats, _ = pp.voxelize(T(pcl[:, :3].copy()), T(pcl[:, [0, 1, 2, 6, 7, 8]].copy()), 50, [1900, 2048, 512])
    assert np.array_equal(locs.cpu().numpy(), g["vox2_locs"])
    np.testing.assert_allclose(feats.cpu().numpy(), g["vox2_feats"], rtol=1e-6, atol=1e-6)
    rs = np.random.RandomState(2)
    pts = rs.uniform(0, 21.7, (1200000, 3)).astype(np.float32)
    f = rs.randn(1200000, 9).astype(np.float32)
    th = 0.3
    m = np.array([[np.cos(th), np.sin(th), 0], [-np.sin(th), np.cos(th), 0], [0, 0, 1]]) * 25.0
    locs, feats, size3d = pp.voxelize(T(pts), T(f), 25, [700, 700, 512], matrix=m, batch_index=3)
    wl, wf, ws = po.voxelize(pts, f, 25, [700, 700, 512], matrix=m)
    assert locs.shape[0] == wl.shape[0] < pts.shape[0] and (locs[:, 3] == 3).all()
    same = (locs[:, :3].cpu().numpy() == wl).all(1)
    assert same.mean() > 0.99999  # (a point within one float64 ulp of a voxel face may fall either way: fused multiply-add vs BLAS)
    np.testing.assert_allclose(feats.cpu().numpy(), wf, rtol=1e-5, atol=1e-5)
    # the voxelised cloud feeds the backbone's InputLayer directly
    scn = _scn()
    x = scn.InputLayer(3, [2048, 2048, 512], mode=4)([locs[:, :3].contiguous(), feats])
    assert x.features.shape[0] == np.unique(wl, axis=0).shape[0]


def test_detector_backbone_rpn_proposals_end_to_end():
    """BASELINE.json config 3: points -> backbone -> RPN head + anchors -> decode + rotated NMS -> proposals, all on the device
    (detector.SparseRPNDetector), against the CPU chain run on the golden outputs of the reference's backbone + RPN head for the same
    building.  The head's raw outputs are scaled as in tests/golden/make_golden_postproc.py (random weights); fp32 mode, so the ranking of
    the candidates and the surviving set are those of the reference's own logits."""
    scn = _scn()
    from detection_3d_b200 import detector, postproc as pp
    from oracle import postproc_oracle as po
    g = np.load(os.path.join(GOLD, "rpn_sw4c_mid.npz"))
    q = np.load(os.path.join(GOLD, "postproc.npz"))
    OS, RS = float(q["obj_scale"]), float(q["reg_scale"])
    anchors, logits, regs = _rpn_golden_inputs()
    try:
        scn.set_math_mode("fp32")
        net = scn.FPN_Net(**scn.sw4c_fpn432_config())
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        det = detector.SparseRPNDetector(net, detector.RPNModule(pre_nms_top_n=200, post_nms_top_n=120, nms_thresh=0.3))
        state = {k[2:]: torch.from_numpy(g[k]).clone() for k in g.files if k.startswith("w:")}
        for k in ("cls_logits", "bbox_pred"):  # fold the scaling into the output layers: the module then produces the scaled outputs itself
            sc = OS if k == "cls_logits" else RS
            state[k + ".weight"] *= sc
            state[k + ".bias"] *= sc
        det.rpn.head.load_state_dict(state)
        det = det.cuda().eval()
        coords = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
        with torch.no_grad():
            groups = det([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert len(groups) == 2 and all(len(gr) == 1 for gr in groups)
    for gi in range(2):
        wb, wo = po.rpn_post_process(anchors, logits[:, gi] * np.float32(OS), regs[:, 7 * gi:7 * gi + 7] * np.float32(RS), 200, 120, 0.3, (0.3, 0.3))
        got = groups[gi][0]
        assert tuple(got.bbox3d.shape) == wb.shape
        _close(got.bbox3d.cpu().numpy(), wb, 3e-3, 3e-4)   # the backbone's fp32 end-to-end tolerance carried through head and decode
        np.testing.assert_allclose(got.get_field("objectness").cpu().numpy(), wo, rtol=3e-3, atol=3e-4)


# ------------------------------------------------------------------ replayed training step: input gradient, misuse
def test_replayed_training_step_input_gradient_and_misuse():
    """The replayed training step (program.TrainFunction) against the layer-by-layer autograd path of the same network: gradient of
    the network INPUT (InputLayer backward through scn_program_backward, gradients brought from the reference's row order into the
    internal one on the way in) and parameter gradients, fp32 mode (summation order only); a second training forward before
    backward() raises instead of using activations that are gone."""
    scn = _scn()
    cfg = dict(fpn_util.mini4_config(), track_running_stats=True)
    coords = synthetic.building_coords(nx=52, ny=44, nz=20, n_walls=3, seed=4)
    feats_np = fpn_util.features_for(coords)
    rs = np.random.RandomState(0)

    def step(net, w):
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net.zero_grad(set_to_none=True)
        f = torch.from_numpy(feats_np).cuda().requires_grad_(True)
        rpn, roi = net([torch.from_numpy(coords), f])
        loss = sum((m.features * wi).sum() for m, wi in zip(rpn + roi, w))
        loss.backward()
        return f.grad.clone(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}, [m.features.detach().clone() for m in rpn + roi]

    try:
        scn.set_math_mode("fp32")
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().train()
        with torch.no_grad():
            net.eval()
            shapes = [m.features.shape for m in sum(net([torch.from_numpy(coords), torch.from_numpy(feats_np).cuda()]), [])]
            net.train()
        w = [torch.from_numpy(rs.randn(*s).astype(np.float32)).cuda() for s in shapes]
        df0, g0, o0 = step(net, w)            # layer by layer (records)
        assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
        n0 = scn.SCN.lib().scn_debug_counter(11)
        df1, g1, o1 = step(net, w)            # replayed
        assert scn.SCN.lib().scn_debug_counter(11) == n0 + 1
        torch.cuda.synchronize()
        for a, b in zip(o0, o1):
            _close(b.cpu().numpy(), a.cpu().numpy(), 2e-3, 2e-4)
        assert set(g0) == set(g1)
        for k in g0:
            _close(g1[k].cpu().numpy(), g0[k].cpu().numpy(), 5e-3, 5e-4)
        _close(df1.cpu().numpy(), df0.cpu().numpy(), 5e-3, 5e-4)
        # misuse: two forwards, then backward of the first
        f = torch.from_numpy(feats_np).cuda()
        rpn_a, _ = net([torch.from_numpy(coords), f])
        net([torch.from_numpy(coords), f])
        with pytest.raises(RuntimeError, match="another forward"):
            rpn_a[0].features.sum().backward()
    finally:
        scn.set_math_mode("fp32")


def test_empty_cache_releases_library_memory_and_forward_still_works():
    """scn.empty_cache() (scn_release_cached_memory): the idle Metadata chunks, weight images and scratch buffers go back to the
    driver; the next forward allocates them again and gives the same result."""
    scn = _scn()
    cfg = fpn_util.mini4_config()
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net = net.cuda().eval()
    coords = synthetic.building_coords(nx=44, ny=40, nz=20, n_walls=3, seed=9)
    x = [torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()]
    with torch.no_grad():
        a = [m.features.clone() for m in sum(net(x), [])]
        a2 = [m.features.clone() for m in sum(net(x), [])]   # replayed
        del a2
        net.reset_program()
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        released = scn.empty_cache()
        free1 = torch.cuda.mem_get_info()[0]
        assert released > 0 and free1 > free0, (released, free0, free1)
        b = [m.features.clone() for m in sum(net(x), [])]
    torch.cuda.synchronize()
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def test_gradient_reducer_attach_writes_replayed_gradients_into_flat_buffer():
    """distributed.GradientReducer.attach: the replayed backward pass writes the parameter gradients straight into the reducer's flat
    buffer (p.grad are views of it) and returns none to autograd; same values as the layer-by-layer step of the same state (fp32)."""
    scn = _scn()
    from detection_3d_b200 import distributed
    cfg = fpn_util.mini4_config()
    coords = synthetic.building_coords(nx=48, ny=44, nz=20, n_walls=3, seed=6)
    feats = torch.from_numpy(fpn_util.features_for(coords)).cuda()
    try:
        scn.set_math_mode("fp32")
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().train()
        red = distributed.GradientReducer([p for p in net.parameters() if p.requires_grad])
        assert not red.attach(net)  # no program yet
        got = []
        for step in range(3):
            if step == 1:
                assert red.attach(net)
            net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
            red.zero()
            rpn, roi = net([torch.from_numpy(coords), feats])
            sum((m.features ** 2).mean() for m in rpn + roi).backward()
            red.finish()
            torch.cuda.synchronize()
            for p in red.params:  # still views of the flat buffer
                lo, hi = red.slices[p]
                assert p.grad.data_ptr() == red.flat.data_ptr() + lo * 4
            got.append(red.flat.clone())
        assert scn.SCN.lib().scn_debug_counter(11) >= 2
    finally:
        scn.set_math_mode("fp32")
    assert float(got[0].abs().max()) > 0
    scale = float(got[0].abs().max())
    for g in got[1:]:
        np.testing.assert_allclose(g.cpu().numpy(), got[0].cpu().numpy(), rtol=5e-3, atol=5e-4 * scale)
