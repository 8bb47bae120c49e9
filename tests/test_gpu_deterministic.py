"""Deterministic mode: under torch.use_deterministic_algorithms(True) every float the library produces is bitwise reproducible from
run to run (include/scn_b200.h, scn_set_deterministic; DESIGN.md section 7).  Each test turns torch's flag on in a fixture and
restores it afterwards.  The "float-atomic launches" counter (scn_debug_counter(14)) proves that no launch accumulated floats in an
order-dependent way; the results stay within the tolerances the other parity tests use against the reference."""
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch

import fpn_util
from detection_3d_b200 import synthetic

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = torch.LongTensor
CNT = dict(stats=4, bn_from_sums=8, split=9, float_atomic=14)
TC_E2E = {"fp32": 2e-3, "tf32": 1e-2, "bf16": 4.5e-2}   # end to end vs the reference's fp32 outputs, max|d| / max(1, max|ref|)
MINI4_BLD = dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)


@pytest.fixture
def det():
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn)


def _scn(math):
    import detection_3d_b200.sparseconvnet as scn
    if math != "fp32" and not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    scn.set_math_mode(math)
    return scn


def _counters():
    from detection_3d_b200._lib import lib
    return {k: lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _inputs(bld=MINI4_BLD, grad=False):
    c = synthetic.building_coords(**bld)
    f = torch.from_numpy(fpn_util.features_for(c)).cuda()
    return torch.from_numpy(c), f.requires_grad_(True) if grad else f


def _net(scn, train=False, cfg=None):
    cfg = cfg or fpn_util.mini4_config()
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    return net.cuda().train() if train else net.cuda().eval()


def _forward(net, inputs):
    with torch.no_grad():
        rpn, roi = net(list(inputs))
    return [m.features.clone() for m in rpn + roi]


def _equal(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and torch.equal(x, y), (i, float((x - y).abs().max()) if x.shape == y.shape else None)


def _train_cfg():
    return dict(fpn_util.mini4_config(), track_running_stats=True)


def _train_step(net, inputs, state=None):
    """one training step: (loss terms, parameter gradients, input gradient, buffers); `state` is loaded first"""
    if state is not None:
        net.load_state_dict(state)
    net.zero_grad(set_to_none=True)
    c, f = inputs
    f = f.detach().clone().requires_grad_(True)
    rpn, roi = net([c, f])
    terms = [(m.features ** 2).mean() for m in rpn + roi]
    sum(terms).backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
    bufs = {k: b.clone() for k, b in net.named_buffers()}
    return torch.stack([t.detach() for t in terms]), grads, f.grad.clone(), bufs


def _same_step(a, b):
    assert torch.equal(a[0], b[0])
    assert a[1].keys() == b[1].keys()
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
    assert torch.equal(a[2], b[2])
    for k in a[3]:
        assert torch.equal(a[3][k], b[3][k]), k


# ------------------------------------------------------------------ 1. no order-dependent atomics
def test_no_float_atomics_in_deterministic_mode(det):
    """bf16 replayed forward of the mini4 golden building, bf16 replayed training step, fp32 layer-by-layer training step: the
    float-atomic counter does not move under the flag, while the split-offset, epilogue-statistics and BatchNorm-from-sums paths
    ran; the same replayed forward without the flag does move it (the counter is wired)."""
    scn = _scn("bf16")
    try:
        net, inputs = _net(scn), _inputs()
        _forward(net, inputs)  # records
        before = _counters()
        _forward(net, inputs)  # replays
        torch.cuda.synchronize()
        d = _delta(before)
        assert d["float_atomic"] == 0 and d["split"] > 0 and d["stats"] > 0 and d["bn_from_sums"] > 0, d
        torch.use_deterministic_algorithms(False)
        before = _counters()
        _forward(net, inputs)
        torch.cuda.synchronize()
        assert _delta(before)["float_atomic"] > 0
        torch.use_deterministic_algorithms(True)

        tnet = _net(scn, train=True, cfg=_train_cfg())
        state = {k: v.clone() for k, v in tnet.state_dict().items()}
        _train_step(tnet, inputs, state)  # records
        assert tnet.__dict__.get("_program_train") is not None, tnet.__dict__.get("_program_train_error")
        before = _counters()
        _train_step(tnet, inputs, state)  # replays
        d = _delta(before)
        assert d["float_atomic"] == 0 and d["split"] > 0, d

        scn.set_math_mode("fp32")
        fnet = _net(scn, train=True, cfg=_train_cfg())
        fnet.__dict__["_program_train_error"] = "layer by layer"  # keeps the network on the layer-by-layer path
        before = _counters()
        _train_step(fnet, inputs)
        assert fnet.__dict__.get("_program_train") is None
        assert _delta(before)["float_atomic"] == 0
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ 2. repeatable forward
@pytest.mark.parametrize("math", ["fp32", "tf32", "bf16"])
def test_repeatable_forward(det, math):
    """Two fresh networks with the same weights give the same recording forward; three replays agree with each other; two replays
    on prefetched Metadata agree with each other; every map stays within the end-to-end bound of the reference's outputs."""
    scn = _scn(math)
    g = np.load(os.path.join(GOLD, "fpn_mini4.npz"))
    try:
        inputs = _inputs()
        a, b = _net(scn), _net(scn)
        rec = _forward(a, inputs)
        _equal(rec, _forward(b, inputs))
        reps = [_forward(a, inputs) for _ in range(3)]
        _equal(reps[0], reps[1])
        _equal(reps[0], reps[2])
        # streaming: a Metadata built ahead by FPN_Net.prefetch is a path of its own (its BatchNorm sums come out in another order
        # than those of a replay that builds its own Metadata); two prefetched replays agree bit for bit
        dev_inputs = (inputs[0].cuda(), inputs[1])
        streamed = []
        for _ in range(2):
            assert a.prefetch(dev_inputs[0])
            streamed.append(_forward(a, dev_inputs))
        _equal(streamed[0], streamed[1])
        keys = [f"rpn{i}" for i in range(int(g["n_rpn"]))] + [f"roi{i}" for i in range(int(g["n_roi"]))]
        for out in (rec, reps[0], streamed[0]):
            for k, x in zip(keys, out):
                ref = g[k + "_features"]
                err = float(np.abs(x.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max()))
                assert err < TC_E2E[math], (k, err)
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ 3. scheduling independence
_CHILD = r"""
import os, sys
import numpy as np, torch
sys.path[:0] = [{root!r}, os.path.join({root!r}, "tests")]
import fpn_util
import detection_3d_b200.sparseconvnet as scn
from detection_3d_b200 import synthetic
torch.use_deterministic_algorithms(True)
scn.set_math_mode("bf16")
out = {out!r}
c = synthetic.building_coords(**{bld!r})
c, f = torch.from_numpy(c), torch.from_numpy(fpn_util.features_for(c)).cuda()
net = scn.FPN_Net(**fpn_util.mini4_config())
net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
net = net.cuda().eval()
with torch.no_grad():
    net([c, f])
    rpn, roi = net([c, f])
for i, m in enumerate(rpn + roi):
    np.save(os.path.join(out, f"fwd{{i}}.npy"), m.features.cpu().numpy())
net = scn.FPN_Net(**dict(fpn_util.mini4_config(), track_running_stats=True))
state = fpn_util.deterministic_state(net, seed=1)
net = net.cuda().train()
for step in range(2):
    net.load_state_dict(state)
    net.zero_grad(set_to_none=True)
    rpn, roi = net([c, f])
    sum((m.features ** 2).mean() for m in rpn + roi).backward()
assert net.__dict__.get("_program_train") is not None
for k, p in net.named_parameters():
    if p.grad is not None:
        np.save(os.path.join(out, "grad_" + k + ".npy"), p.grad.cpu().numpy())
for k, b in net.named_buffers():
    np.save(os.path.join(out, "buf_" + k + ".npy"), b.cpu().numpy())
"""


def test_results_do_not_depend_on_scheduling(tmp_path):
    """The bf16 replayed forward and one bf16 replayed training step in three processes: default work distribution, the atomic
    work counter (SCN_TC_DYNAMIC=1) and a smaller grid (SCN_TC_SMS=37).  Outputs, gradients and running statistics are bitwise
    equal: partial sums are indexed by work item, not by the CTA that happened to compute them."""
    import detection_3d_b200.sparseconvnet as scn
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    dirs = []
    for name, extra in (("default", {}), ("dynamic", {"SCN_TC_DYNAMIC": "1"}), ("sms37", {"SCN_TC_SMS": "37"})):
        d = tmp_path / name
        d.mkdir()
        env = dict(os.environ, **extra)
        r = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, out=str(d), bld=MINI4_BLD)], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (name, r.stderr[-3000:])
        dirs.append(d)
    names = sorted(os.listdir(dirs[0]))
    assert any(n.startswith("fwd") for n in names) and any(n.startswith("grad_") for n in names)
    for d in dirs[1:]:
        assert sorted(os.listdir(d)) == names
        for n in names:
            a, b = np.load(dirs[0] / n), np.load(d / n)
            assert a.shape == b.shape and a.tobytes() == b.tobytes(), (d.name, n)


# ------------------------------------------------------------------ 4. repeatable training step
@pytest.mark.parametrize("math", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("replay", [False, True])
def test_repeatable_training_step(det, math, replay):
    """The setup of test_whole_network_training_step_vs_reference_autograd, state reloaded before each step: two steps give
    bitwise equal parameter gradients, input-feature gradients, loss terms and running statistics (which carry saveMean /
    saveInvStd), within that test's bounds of the reference's step (fpn_mini4_train.npz)."""
    scn = _scn(math)
    g = np.load(os.path.join(GOLD, "fpn_mini4_train.npz"))
    tol_max, tol_rms = {"fp32": (5e-3, 5e-3), "tf32": (2.5e-1, 8e-2), "bf16": (5e-1, 2e-1)}[math]
    tol = {"fp32": 5e-3, "tf32": 3e-2, "bf16": 8e-2}[math]
    try:
        net, inputs = _net(scn, train=True, cfg=_train_cfg()), _inputs()
        state = {k: v.clone() for k, v in net.state_dict().items()}
        if replay:
            _train_step(net, inputs, state)  # records
            assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
        else:
            net.__dict__["_program_train_error"] = "layer by layer"
        first = _train_step(net, inputs, state)
        second = _train_step(net, inputs, state)
        assert (net.__dict__.get("_program_train") is not None) == replay
    finally:
        scn.set_math_mode("fp32")
    _same_step(first, second)
    np.testing.assert_allclose(first[0].cpu().numpy(), g["map_mean_sq"], rtol=tol)
    want = {k[5:] for k in g.files if k.startswith("grad:")}
    assert set(first[1]) == want
    for k in want:
        ref = g["grad:" + k].astype(np.float64)
        d = first[1][k].cpu().numpy().astype(np.float64) - ref
        assert np.abs(d).max() / max(1e-6, np.abs(ref).max()) < tol_max, k
        assert np.sqrt((d * d).mean()) / max(1e-12, np.sqrt((ref * ref).mean())) < tol_rms, k
    for k, b in first[3].items():
        ref = g["buf:" + k]
        np.testing.assert_allclose(b.cpu().numpy(), ref, rtol=tol, atol=tol * max(1e-3, float(np.abs(ref).max())), err_msg=k)


# ------------------------------------------------------------------ 5. per-op repeatability at shapes that hit every site
def _twice_and_default(fn):
    """fn() twice under the flag (bitwise equal) and once without it; returns (deterministic result, default result)"""
    a, b = fn(), fn()
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    torch.use_deterministic_algorithms(False)
    try:
        c = fn()
    finally:
        torch.use_deterministic_algorithms(True)
    return a, c


def _close(got, want, rtol, atol):
    want = want.double().cpu()
    scale = max(1.0, float(want.abs().max())) if want.numel() else 1.0
    np.testing.assert_allclose(got.double().cpu().numpy(), want.numpy(), rtol=rtol, atol=atol * scale)


@pytest.mark.parametrize("C", [64, 30])
def test_batchnorm_forward_backward_large(det, C):
    """Standalone BatchNorm with n = 300 000 rows (the multi-CTA statistics kernels, float4 and scalar): saveMean / saveInvStd,
    running statistics, output, input / weight / bias gradients, against a float64 restatement."""
    import detection_3d_b200.sparseconvnet as scn
    rs = np.random.RandomState(C)
    n = 300000
    x = torch.from_numpy((rs.randn(n, C) * 2 + 0.5).astype(np.float32)).cuda()
    dy = torch.from_numpy(rs.randn(n, C).astype(np.float32)).cuda()
    w = torch.from_numpy((1 + 0.1 * rs.randn(C)).astype(np.float32)).cuda()
    b = torch.from_numpy((0.1 * rs.randn(C)).astype(np.float32)).cuda()

    def run():
        out, sm, si = torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        scn.SCN.BatchNormalization_updateOutput(x, out, sm, si, rm, rv, w, b, 1e-4, 0.9, True, 0.0)
        dx, dw, db, d = torch.empty(0, device="cuda"), torch.empty(C, device="cuda"), torch.empty(C, device="cuda"), dy.clone()
        scn.SCN.BatchNormalization_backward(x, dx, out, d, sm, si, rm, rv, w, b, dw, db, 0.0)
        torch.cuda.synchronize()
        return out, sm, si, rm, rv, dx, dw, db
    got, _ = _twice_and_default(run)
    out, sm, si, rm, rv, dx, dw, db = got
    xd = x.double()
    mean, var = xd.mean(0), xd.var(0, unbiased=False)
    inv = (var + 1e-4) ** -0.5
    y = (xd - mean) * inv * w.double() + b.double()
    _close(sm, mean, 1e-5, 1e-6)
    _close(si, inv, 1e-5, 1e-6)
    _close(rv, 0.9 + 0.1 * xd.var(0, unbiased=True), 1e-5, 1e-6)
    _close(out, y.clamp(min=0), 1e-4, 1e-5)
    dd = dy.double() * (y > 0)
    _close(db, dd.sum(0), 1e-4, 1e-5)
    _close(dw, (dd * (xd - mean) * inv).sum(0), 1e-4, 1e-5)
    dxw = (dd - dd.mean(0) - (xd - mean) * inv * inv * (dd * (xd - mean)).mean(0)) * inv * w.double()
    _close(dx, dxw, 1e-4, 1e-5)


def _grid(scn, bld, sz):
    from gpu_adapter import GpuMetadata
    G = GpuMetadata()
    G.input_layer(sz, synthetic.building_coords(**bld), 0, 4)
    return G, G.nactive(sz)


@pytest.mark.parametrize("case", ["split_cout256", "dw_tc_parts", "k_dw_fp32", "k_dw_tf32"])
def test_convolution_sites(det, case):
    """split_cout256: a bf16 submanifold convolution 64 -> 256 on a level of <= 40 work items (filter offsets split over CTAs);
    dw_tc_parts: the bf16 tensor-core weight gradient of a 128 -> 128 layer whose rule lists are cut into several parts;
    k_dw_*: the CUDA-core weight gradient (fp32, tf32).  Twice bitwise under the flag, and within the per-layer tolerance of the
    default mode's result (which the parity tests pin to the reference)."""
    math = {"split_cout256": "bf16", "dw_tc_parts": "bf16", "k_dw_fp32": "fp32", "k_dw_tf32": "tf32"}[case]
    scn = _scn(math)
    try:
        if case == "split_cout256":
            sz, bld, cin, cout = [32, 32, 16], dict(nx=24, ny=20, nz=10, n_walls=2, seed=1), 64, 256
        elif case == "dw_tc_parts":
            sz, bld, cin, cout = [256, 256, 64], dict(nx=200, ny=180, nz=40, n_walls=4, seed=2), 128, 128
        else:
            sz, bld, cin, cout = [64, 64, 32], dict(nx=40, ny=36, nz=12, n_walls=3, seed=4), 32, 64
        G, n = _grid(scn, bld, sz)
        if case == "split_cout256":
            assert n <= 40 * 128
        rs = np.random.RandomState(7)
        x = torch.from_numpy(rs.randn(n, cin).astype(np.float32)).cuda()
        w = torch.from_numpy((rs.randn(27, 1, cin, cout) * (2.0 / (cin * 27)) ** 0.5).astype(np.float32)).cuda()
        dy = torch.from_numpy(rs.randn(n, cout).astype(np.float32)).cuda()

        def run():
            before = _counters()
            out = torch.empty(0, device="cuda")
            scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([3, 3, 3]), G.m, x, out, w, torch.Tensor())
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            scn.SCN.SubmanifoldConvolution_backward(L(sz), L([3, 3, 3]), G.m, x, din, dy, w, dw, torch.Tensor())
            torch.cuda.synchronize()
            d = _delta(before)
            if torch.are_deterministic_algorithms_enabled():
                assert d["float_atomic"] == 0, d
            if case == "split_cout256":
                assert d["split"] > 0, d
            return out, din, dw
        got, dflt = _twice_and_default(run)
        rtol, atol = {"fp32": (1e-4, 1e-5), "tf32": (4e-3, 2e-3), "bf16": (1.6e-2, 8e-3)}[math]
        for a, b in zip(got, dflt):
            _close(a, b, rtol, atol)
    finally:
        scn.set_math_mode("fp32")


def test_network_in_network_backward_with_bias(det):
    """NetworkInNetwork backward with a bias: weight and bias gradients from per-chunk partials, twice bitwise, and within fp32
    rounding of the default mode's result."""
    scn = _scn("fp32")
    rs = np.random.RandomState(3)
    n, cin, cout = 50000, 64, 96
    x = torch.from_numpy(rs.randn(n, cin).astype(np.float32)).cuda()
    dy = torch.from_numpy(rs.randn(n, cout).astype(np.float32)).cuda()
    m = scn.NetworkInNetwork(cin, cout, True).cuda()

    def run():
        m.zero_grad(set_to_none=True)
        xt = x.clone().requires_grad_(True)
        y = m(scn.SparseConvNetTensor(features=xt, metadata=None, spatial_size=L([8, 8, 8]))).features
        before = _counters()
        y.backward(dy)
        torch.cuda.synchronize()
        if torch.are_deterministic_algorithms_enabled():
            assert _delta(before)["float_atomic"] == 0
        return m.weight.grad.clone(), m.bias.grad.clone(), xt.grad.clone()
    got, dflt = _twice_and_default(run)
    for a, b in zip(got, dflt):
        _close(a, b, 1e-4, 1e-5)


# ------------------------------------------------------------------ 6. toggling
def test_toggling_leaves_no_stale_state(det):
    """on -> off -> on: the second deterministic replay gives the bits of the first."""
    scn = _scn("bf16")
    try:
        net, inputs = _net(scn), _inputs()
        _forward(net, inputs)
        first = _forward(net, inputs)
        torch.use_deterministic_algorithms(False)
        _forward(net, inputs)
        torch.use_deterministic_algorithms(True)
        _equal(first, _forward(net, inputs))
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ 7. alerts
def test_roi_align_backward_alerts(det):
    """ROIAlignRotated3D backward has no deterministic implementation: it raises under the flag and warns in warn-only mode (with
    the result of the default mode, to 1e-5); the forward is unaffected."""
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200.roi_align import ROIAlignRotated3D
    coords = synthetic.small_building(20, 18, 8, 2, seed=4)
    rs = np.random.RandomState(5)
    sz = [32, 32, 8]
    rois = torch.tensor([[0, 8, 9, 3, 6, 5, 3, 30], [0, 14, 6, 4, 4, 7, 2, -60]], dtype=torch.float32, device="cuda")
    feats = torch.from_numpy(rs.randn(coords.shape[0], 12).astype(np.float32)).cuda()
    g = torch.from_numpy(rs.randn(2, 12, 3, 4, 2).astype(np.float32)).cuda()

    def run():
        ft = feats.clone().requires_grad_(True)
        x = scn.InputLayer(3, sz, mode=4)([torch.from_numpy(coords.astype(np.int64)), ft])
        out = ROIAlignRotated3D((3, 4, 2), 1.0, 2)(x, rois)
        return out, ft
    out, ft = run()
    with pytest.raises(RuntimeError, match="ROIAlignRotated3D backward"):
        out.backward(g)
    torch.use_deterministic_algorithms(True, warn_only=True)
    out2, ft2 = run()
    assert torch.equal(out, out2)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        out2.backward(g)
    assert any("ROIAlignRotated3D backward" in str(r.message) for r in rec)
    torch.use_deterministic_algorithms(False)
    out3, ft3 = run()
    assert torch.equal(out, out3)
    out3.backward(g)
    torch.cuda.synchronize()
    np.testing.assert_allclose(ft2.grad.cpu().numpy(), ft3.grad.cpu().numpy(), rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------ 8. config 3 end to end
def test_detector_proposals_repeatable(det):
    """BASELINE.json config 3 (voxeliser excluded: integer work) -- backbone, RPN head, anchors, decode, rotated NMS -- runs under
    torch.use_deterministic_algorithms(True) without raising, and two calls give the same boxes, scores and keep counts."""
    scn = _scn("bf16")
    from detection_3d_b200 import detector
    try:
        net = scn.FPN_Net(**scn.sw4c_fpn432_config())
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        d = detector.SparseRPNDetector(net, detector.RPNModule(pre_nms_top_n=200, post_nms_top_n=120, nms_thresh=0.3)).cuda().eval()
        inputs = _inputs(dict(nx=300, ny=280, nz=40, n_walls=5, seed=5))
        runs = []
        for _ in range(3):  # the first call records the backbone's program, the others replay it
            with torch.no_grad():
                groups = d(list(inputs))
            torch.cuda.synchronize()
            runs.append([(b.bbox3d.clone(), b.get_field("objectness").clone()) for gr in groups for b in gr])
        for other in runs[2:]:
            assert len(other) == len(runs[1])
            for (ba, sa), (bb, sb) in zip(runs[1], other):
                assert ba.shape == bb.shape and torch.equal(ba, bb) and torch.equal(sa, sb)
        assert all(b.shape[0] > 0 for b, _ in runs[1])
    finally:
        scn.set_math_mode("fp32")
