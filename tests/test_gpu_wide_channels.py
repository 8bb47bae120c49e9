"""Convolutions wider than 256 channels on the tensor cores (DESIGN.md sections 4.4, 4.6 and 7).

A layer of 256 < Cout <= 1024 output channels (a multiple of 32) runs as ceil(Cout / 256) launches of the unchanged conv_plan_tc over
column slabs of balanced widths, each writing its columns of the full-width rows; the input gradient of a layer with Cin > 256 is
such a launch with Cin and Cout swapped; the weight gradient of a layer wider than 256 on either side runs conv_dw_tc once per
channel block (bf16 / fp16 modes).  scn_debug_counter(10) counts CUDA-core convolution launches and scn_debug_counter(21) the
CUDA-core weight-gradient kernel k_dw, so every tensor-core case below proves the tensor-core paths ran.

Exact grid as in test_gpu_tc_exact.py: forward, input gradient and weight gradient bit for bit against the fp64 gather-GEMM in every
math mode; the fused epilogue across slabs; per-layer tolerances on N(0, 1) data; deterministic mode; FPN_Net end to end with wide
levels, and its replayed training step."""
import ctypes as C

import numpy as np
import pytest
import torch

import fpn_util
import test_gpu_large_filters as lf
import test_gpu_tc_exact as tx
from detection_3d_b200 import synthetic

MODES = dict(tx.MODES, fp16=5)  # (tx.MODES has the four modes before fp16)
TC_MODES = ("tf32", "bf16", "tf32x3", "fp16")
CNT = dict(tx.CNT, chunk=16, train_replay=11, half_only=5, f16=18, k_dw=21)
# per layer on N(0, 1) data: rtol, atol x max|ref| (DESIGN.md section 7; fp16 as test_gpu_fp16.py)
LAYER_TOL = dict(lf.LAYER_TOL, fp16=(2e-3, 1e-3))


def _counters():
    return {k: tx._lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _set_mode(mode):
    tx._check(tx._lib().scn_set_math_mode(MODES[mode]))


def _level_geom(kind, level, shape):
    """(level, geometry) -- shape: a filter volume of test_gpu_tc_exact (27 = 3^3, 8 = 2^3 / 2, 16 = z-collapse, 1 = NiN) or a
    filter name of test_gpu_large_filters ("5" = 5^3)"""
    if isinstance(shape, str):
        lv = lf._wlevel(level)
        return lv, lf._wgeom(lv, kind, shape)
    lv = tx._level(level)
    return lv, dict(tx._geom(lv, kind, shape), K=shape)


def _inputs(case, seed=0):
    kind, level, shape, cin, cout = case
    rs = np.random.RandomState(seed + 7 * cin + 13 * cout + sum(map(ord, kind + level + str(shape))))
    lv, g = _level_geom(kind, level, shape)
    x = tx.grid_x(rs, g["n_src"], cin)
    w = tx.grid_w(rs, cin, cout) if kind == "nin" else tx.grid_w(rs, g["K"], cin, cout)
    dy = tx.grid_w(rs, g["n_dst"], cout)
    return lv, g, x, w, dy


# ------------------------------------------------------------------ 1. exact grid, bit for bit
CASES = [
    ("subm", "small", 27, 64, 288), ("subm", "mini4", 27, 256, 512), ("subm", "rows129", 27, 512, 512), ("subm", "big", 27, 512, 256),
    ("subm", "rows1", 27, 320, 384), ("subm", "mini4", 27, 32, 1024),
    ("conv", "small", 8, 256, 512),     # strided 2^3 / 2
    ("deconv", "mini4", 8, 512, 288),   # 2^3 / 2, one parent per fine site
    ("conv", "small", 16, 288, 288),    # z-collapse [1, 1, z]
    ("subm", "small", "5", 64, 320),    # 5^3: two offset chunks, each in two slabs
    ("nin", "mini4", 1, 512, 384),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=tx._cid)
@pytest.mark.parametrize("mode", list(MODES))
def test_exact_grid_bitwise(mode, case):
    """Forward, input gradient and weight gradient equal the fp64 reference bit for bit.  In the tensor-core modes no convolution,
    forward or input gradient, runs on the CUDA cores; in bf16 / fp16 no weight gradient does either."""
    if mode != "fp32":
        tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv, g, x, w, dy = _inputs(case)
    want = tx.ref_forward(lv, kind, g, x, w)
    tc = mode != "fp32"
    try:
        _set_mode(mode)
        before = _counters()
        out, _ = tx.run_forward(lv, kind, g, x, w)
        d = _delta(before)
        print(f"[wide ch] {mode} {tx._cid(case)} forward: {d}")
        tx.assert_exact(out, want, f"{mode} {tx._cid(case)} forward")
        if tc:
            assert d["simt"] == 0 and d["tc"] >= -(-cout // 256), d
            assert (d["x3"] > 0) == (mode == "tf32x3"), d
            assert (d["f16"] > 0) == (mode == "fp16" and cin % 64 == 0), d  # (32-channel rows keep TF32 operands)
        else:
            assert d["tc"] == 0 and d["simt"] > 0, d
        if kind == "nin":
            return
        before = _counters()
        d_in, dw = tx.run_backward(lv, kind, g, x, dy, w)
        d = _delta(before)
        print(f"[wide ch] {mode} {tx._cid(case)} backward: {d}")
        want_din, want_dw = tx.ref_backward(lv, kind, g, x, dy, w)
        tx.assert_exact(d_in, want_din, f"{mode} {tx._cid(case)} input gradient")
        tx.assert_exact(dw, want_dw, f"{mode} {tx._cid(case)} weight gradient")
        if tc:
            assert d["simt"] == 0, d
            assert (d["k_dw"] == 0) == (mode in ("bf16", "fp16")), d
            if mode == "fp16":
                assert d["f16"] > 0, d
    finally:
        _set_mode("fp32")


# ------------------------------------------------------------------ 2. fused epilogue across slabs
def _copy16(t, mode):
    return t.half() if mode == "fp16" else t.to(torch.bfloat16)


@pytest.mark.gpu
@pytest.mark.parametrize("c_lat", [32, 128])
@pytest.mark.parametrize("case", [("subm", "mini4", 27, 64, 288), ("subm", "small", 27, 128, 512), ("deconv", "small", 8, 256, 288)],
                         ids=tx._cid)
@pytest.mark.parametrize("mode", TC_MODES)
def test_fused_epilogue_across_slabs(mode, case, c_lat):
    """Bias, the caller's addend, the 16-bit copy (equal to out converted) and the lateral stage y[row] @ W_lat, each slab taking its
    columns of every one; rows past the output stay untouched.  The statistics request (more than 128 channels) is reported as not
    taken.  The small building splits its offsets over CTAs: the zeroing, atomics and 16-bit pass cover the slab's columns only."""
    tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv, g, x, w, _ = _inputs(case, seed=1)
    n = g["n_dst"]
    rs = np.random.RandomState(cin + cout + c_lat)
    b = tx.grid_w(rs, cout) if kind != "deconv" else None  # (a deconvolution with bias takes the CUDA-core path)
    ad = tx.grid_w(rs, n, cout)
    y, wl = tx.grid_x(rs, n, c_lat, 0.1), tx.grid_w(rs, c_lat, cout)
    want = tx.ref_forward(lv, kind, g, x, w, b, ad) + y.double() @ wl.double()
    y16 = _copy16(y, mode)  # (kept alive until the launch has read it)
    lib = tx._lib()
    try:
        _set_mode(mode)
        stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
        before = _counters()
        tx._check(lib.scn_fuse_next_lateral(tx._p(y), tx._p(y16), tx._p(wl), 0, c_lat, n))
        tx._check(lib.scn_fuse_next_stats(tx._p(stats)))
        out, o16 = tx.run_forward(lv, kind, g, x, w, b, ad, want16=True)
        took_l, took_s = C.c_int(), C.c_int()
        tx._check(lib.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
        d = _delta(before)
    finally:
        _set_mode("fp32")
    print(f"[wide ch epilogue] {mode} {tx._cid(case)} c_lat={c_lat}: {d}, lateral {took_l.value} stats {took_s.value}")
    assert d["simt"] == 0 and d["tc"] >= 2, d
    assert took_l.value == 1 and d["lateral"] == d["tc"], d  # every slab carried its columns of the lateral stage
    assert took_s.value == 0 and d["stats"] == 0, d
    assert float(stats.abs().sum()) == 0.0
    tx.assert_exact(out, want, f"{mode} {tx._cid(case)} epilogue")
    assert torch.equal(o16.view(torch.int16), _copy16(out, mode).view(torch.int16)), "16-bit copy differs from out converted"


# ------------------------------------------------------------------ 3. per layer on N(0, 1) data
@pytest.mark.gpu
@pytest.mark.parametrize("case", [("subm", "mini4", 27, 256, 512), ("subm", "small", 27, 512, 320), ("conv", "small", 8, 256, 512),
                                  ("deconv", "mini4", 8, 512, 288), ("nin", "mini4", 1, 512, 384)], ids=tx._cid)
@pytest.mark.parametrize("mode", list(MODES))
def test_layer_tolerance_random(mode, case):
    if mode != "fp32":
        tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv, g = _level_geom(kind, level, shape)
    gen = torch.Generator(device="cuda").manual_seed(cin + cout)
    x = torch.randn(g["n_src"], cin, device="cuda", generator=gen)
    k = 1 if kind == "nin" else g["K"]
    w = torch.randn(k, cin, cout, device="cuda", generator=gen) / np.sqrt(cin * k)
    w = w[0] if kind == "nin" else w
    want = tx.ref_forward(lv, kind, g, x, w)
    try:
        _set_mode(mode)
        out, _ = tx.run_forward(lv, kind, g, x, w)
    finally:
        _set_mode("fp32")
    rtol, atol = LAYER_TOL[mode]
    err = (out.double() - want).abs()
    bound = rtol * want.abs() + atol * float(want.abs().max())
    print(f"[wide ch tol] {mode} {tx._cid(case)}: max err {float(err.max()):.3e} of max|ref| {float(want.abs().max()):.3e}")
    assert bool((err <= bound).all()), float((err - bound).max())


# ------------------------------------------------------------------ 4. deterministic mode
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_deterministic_mode(mode):
    """Two runs of forward and backward are bitwise equal with no float-atomic launch, on a level whose offsets are split over CTAs
    (k_split_sum over a slab's columns) and on wide weight gradients in channel blocks."""
    if mode != "fp32":
        tx._tc_or_skip()
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        _set_mode(mode)
        for case in (("subm", "small", 27, 64, 288), ("subm", "mini4", 27, 320, 384), ("deconv", "mini4", 8, 512, 288)):
            kind = case[0]
            rs = np.random.RandomState(3)
            lv, g, _, _, _ = _inputs(case)
            x = torch.from_numpy(rs.randn(g["n_src"], case[3]).astype(np.float32)).cuda()
            w = torch.from_numpy(rs.randn(g["K"], case[3], case[4]).astype(np.float32) / 20).cuda()
            dy = torch.from_numpy(rs.randn(g["n_dst"], case[4]).astype(np.float32)).cuda()
            runs = []
            before = _counters()
            for _ in range(2):
                out, _ = tx.run_forward(lv, kind, g, x, w)
                d_in, dw = tx.run_backward(lv, kind, g, x, dy, w)
                runs.append((out.clone(), d_in.clone(), dw.clone()))
            d = _delta(before)
            print(f"[wide ch det] {mode} {tx._cid(case)}: {d}")
            assert d["atomic"] == 0, (case, d)
            if mode == "bf16" and case[1] == "small":
                assert d["split"] > 0, d
            for a, b in zip(*runs):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), case
    finally:
        _set_mode("fp32")
        torch.use_deterministic_algorithms(on, warn_only=warn)


# ------------------------------------------------------------------ 5. FPN_Net end to end
MINI4_BLD = dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)


def _wide_config(**kw):
    return dict(fpn_util.mini4_config(), nPlanesF=[32, 128, 320, 512], nPlaneM=288, **kw)


def _fpn_inputs():
    coords = synthetic.building_coords(**MINI4_BLD)
    return coords, fpn_util.features_for(coords)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_fpn_wide_channels_end_to_end(mode):
    """Recording forward and two replays of a mini4 FPN_Net with 320-, 512- and 288-channel levels against the oracle port, within
    the end-to-end bounds of test_gpu_large_filters.py (fp16: 8e-3 as test_gpu_fp16.py).  In bf16 / fp16 the replays launch no
    CUDA-core convolution and the program keeps some BatchNorm outputs as 16-bit copies only."""
    if mode != "fp32":
        tx._tc_or_skip()
    import detection_3d_b200.sparseconvnet as scn
    from oracle import fpn_oracle
    cfg = _wide_config()
    net = scn.FPN_Net(**cfg)
    state = fpn_util.deterministic_state(net, seed=1)
    net.load_state_dict(state)
    net = net.cuda().eval()
    coords, feats = _fpn_inputs()
    orpn, oroi, _ = fpn_oracle.run_fpn_port(cfg, state, coords, feats)
    rtol, atol = {"fp32": (2e-3, 2e-4), "tf32x3": (2e-3, 2e-4), "tf32": (0, 3e-2), "bf16": (0, 6e-2), "fp16": (0, 8e-3)}[mode]
    try:
        scn.set_math_mode(mode)
        for rep in range(3):  # records, then replays
            before = _counters()
            with torch.no_grad():
                rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats).cuda()])
            torch.cuda.synchronize()
            d = _delta(before)
            print(f"[wide ch fpn] {mode} pass {rep}: {d}")
            for a, b in zip(rpn + roi, orpn + oroi):
                assert np.array_equal(a.get_spatial_locations().numpy(), b["locations"]), rep
                ref = b["features"]
                got = a.features.cpu().numpy()
                np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol * max(1.0, float(np.abs(ref).max())), err_msg=f"pass {rep}")
            if rep > 0 and mode in ("bf16", "fp16"):
                assert d["simt"] == 0 and d["half_only"] > 0, d
        assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32x3", "bf16"])
def test_fpn_wide_channels_replayed_training_step(mode):
    """The replayed training step (scn_program_run in training mode + scn_program_backward) against the layer-by-layer fp32-mode step
    of the same network.  tf32x3: loss and every parameter gradient within the fp32-class bounds of
    test_gpu_large_filters.test_fpn_wide_filters_replayed_training_step (5e-3); bf16: the worst-element (5e-1 of max|grad|), cosine
    (0.995) and loss (3e-2) bounds of the bf16 training-step tests against the reference's autograd, relative rms per gradient 3e-1
    (measured on an NVIDIA B200, 1000 W: 1.4e-1 and 1.7e-1 in two runs, in the first layer's weight gradient, which collects the bf16 rounding of every
    output-gradient copy above it), and no weight gradient on the CUDA cores."""
    tx._tc_or_skip()
    import detection_3d_b200.sparseconvnet as scn
    cfg = _wide_config(track_running_stats=True)
    coords, feats = _fpn_inputs()
    inp = lambda: [torch.from_numpy(coords), torch.from_numpy(feats).cuda()]

    def step(net):
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net.zero_grad(set_to_none=True)
        rpn, roi = net(inp())
        loss = sum((m.features ** 2).mean() for m in rpn + roi)
        loss.backward()
        torch.cuda.synchronize()
        return float(loss), {k: p.grad.detach().double().cpu() for k, p in net.named_parameters() if p.grad is not None}

    net32 = scn.FPN_Net(**cfg).cuda().train()
    loss32, g32 = step(net32)
    try:
        scn.set_math_mode(mode)
        net = scn.FPN_Net(**cfg).cuda().train()
        step(net)  # records the training program
        assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
        before = _counters()
        loss, g = step(net)
        d = _delta(before)
    finally:
        scn.set_math_mode("fp32")
    print(f"[wide ch train] {mode}: {d}")
    assert d["train_replay"] == 1 and d["simt"] == 0, d
    tol_max, tol_rms, tol_loss = (5e-3, float("inf"), 5e-3) if mode == "tf32x3" else (5e-1, 3e-1, 3e-2)
    if mode == "tf32x3":
        assert d["x3"] > 0, d
    else:
        assert d["k_dw"] == 0, d
    assert set(g) == set(g32)
    errs = {}
    for k in g32:
        dd = g[k] - g32[k]
        errs[k] = (float(dd.abs().max() / max(1e-6, float(g32[k].abs().max()))),
                   float(dd.pow(2).mean().sqrt() / max(1e-12, float(g32[k].pow(2).mean().sqrt()))))
    keys = sorted(g32)
    a = torch.cat([g[k].ravel() for k in keys])
    b = torch.cat([g32[k].ravel() for k in keys])
    cos = float(a @ b / (a.norm() * b.norm()))
    print(f"[wide ch train] {mode}: worst gradient error {max(e[0] for e in errs.values()):.3e} of max|grad|, worst relative rms "
          f"{max(e[1] for e in errs.values()):.3e}, cosine {cos:.6f}, loss {loss:.6g} vs {loss32:.6g}")
    for k, (err, rms) in errs.items():
        assert err < tol_max and rms < tol_rms, (k, err, rms)
    assert cos >= 0.995, cos
    assert abs(loss - loss32) <= tol_loss * loss32
