"""Math mode 'fp16' (scn.set_math_mode, code 5): the tcgen05 gather-GEMM with fp16 operands wherever 'bf16' mode has bf16 ones
(same kind::f16 instruction, only the A / B format field of the instruction descriptor differs), everything else as in 'bf16' mode.
scn_debug_counter(18) counts the launches with fp16 operands (conv_plan_tc and the weight-gradient kernels): every case below
proves with it that the fp16 kernels ran.

1. the mode code; 2. the exact grid of test_gpu_tc_exact.py bit for bit against the fp64 gather-GEMM (activations in {-1, 0, 1},
weights, gradients, bias and addend in {k/8}: all exact in fp16), so a wrongly formatted operand anywhere fails; 3. the operand
convention (round to nearest even, subnormals kept, overflow to inf); 4. per layer on random data and the accumulation-error bound;
5. end to end against the reference's outputs; 6. the training step, loss scaling and torch.amp.GradScaler; 7. switching between
'bf16' and 'fp16'; 8. deterministic mode.  DESIGN.md section 7 states the tolerances and the measured values."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import fpn_util
import test_gpu_tc_exact as tx
from detection_3d_b200 import synthetic

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CNT = dict(tx.CNT, chunk=16, train_replay=11, f16=18)
F16, BF16, FP32 = 5, 2, 0
MINI4_BLD = dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)
MID_BLD = dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)
# per layer, N(0, 1) activations and He-scaled weights: rtol and atol x max|ref|.  Started from tf32's bounds (4e-3, 2e-3) and
# tightened to the measured error with margin: measured on an NVIDIA B200 (1000 W) 2.8-3.5e-4 x max|ref| (DESIGN.md section 7)
LAYER_RTOL, LAYER_ATOL = 2e-3, 1e-3
# end to end: max|got - ref| / max(1, max|ref|) per returned map; tf32's bound is 1e-2, measured mini4 <= 1.5e-3, sw4c_mid <= 4.0e-3
E2E = 8e-3


def _lib():
    return tx._lib()


def _counters():
    return {k: _lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _mode(code):
    tx._check(_lib().scn_set_math_mode(code))


def _scn():
    import detection_3d_b200.sparseconvnet as scn
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    return scn


def run_forward(lv, kind, g, x, w, bias=None, addend=None, want16=False):
    """tx.run_forward with the 16-bit output copy in fp16 (the format of the current mode)"""
    lib = _lib()
    n_in, cin = x.shape
    cout, n = w.shape[-1], g["n_dst"]
    xb = tx._guarded(x, float("nan"))
    ob = torch.full((n + tx.GUARD, cout), tx.SENT, device="cuda")
    o16 = torch.full((n + tx.GUARD, cout), tx.SENT, dtype=torch.float16, device="cuda") if want16 else None
    macs = C.c_double()
    h = lv.G.m._h
    p = tx._p
    if kind == "nin":
        assert addend is None and not want16
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        tx._check(lib.scn_network_in_network_forward(p(xb), p(ob), p(w), p(bias), n_in, cin, cout, C.byref(macs), stream, None, 0))
    else:
        args = (p(xb), p(ob), p(w), p(bias), cin, cout, C.byref(macs), None, 0, p(addend), p(o16))
        if kind == "subm":
            tx._check(lib.scn_submanifold_convolution_forward(h, tx._l3(g["a"]), tx._l3(g["f"]), *args))
        elif kind == "conv":
            tx._check(lib.scn_convolution_forward(h, tx._l3(g["a"]), tx._l3(g["b"]), tx._l3(g["f"]), tx._l3(g["s"]), *args))
        else:
            tx._check(lib.scn_deconvolution_forward(h, tx._l3(g["b"]), tx._l3(g["a"]), tx._l3(g["f"]), tx._l3(g["s"]), *args))
    torch.cuda.synchronize()
    tx._tail_untouched(ob, n, "forward output")
    if want16:
        tx._tail_untouched(o16, n, "fp16 output copy")
    return ob[:n], (o16[:n] if want16 else None)


def _same16(o16, out):
    assert torch.equal(o16.view(torch.int16), out.half().view(torch.int16)), "fp16 copy differs from out.half()"


def _f16_forward(kind, K, cin, cout):
    """whether the forward launch has fp16 operands (launch_conv_plan_tc: 16-bit where bf16 mode has bf16, TF32 elsewhere)"""
    if not tx._expect_tc("bf16", kind, K, cout):
        return False
    pack = kind != "deconv" and cout <= 128
    if pack and cin % 32 and cin != 16:
        return True  # 16-bit rows zero-padded to 16 / 32 / a multiple of 64 channels
    if cin % 32 and not (pack and cin == 16):
        cin = (cin + 31) // 32 * 32  # fp32 rows zero-padded to a multiple of 32
    return cin % 64 == 0 or (pack and cin in (16, 32))


# ------------------------------------------------------------------ 1. the mode code
def test_mode_code():
    scn = _scn()
    lib = _lib()
    try:
        scn.set_math_mode("fp16")
        assert scn.SCN.math_mode() == 5 and lib.scn_get_math_mode() == 5
        for bad in (4, 6):
            assert lib.scn_set_math_mode(bad) != 0 and lib.scn_get_math_mode() == 5
            assert b"fp16" in lib.scn_last_error() and b"5" in lib.scn_last_error()
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ 2. exact grid, bit for bit
@pytest.mark.parametrize("case", tx.FWD_CASES, ids=tx._cid)
def test_exact_grid_bitwise(case):
    """Forward, input gradient and weight gradient of one layer in fp16 mode equal the fp64 reference bit for bit, after a
    256-channel layer has filled the scratch buffers with non-zero data (as in tx.test_exact_grid_bitwise)."""
    tx._tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, dy = tx._inputs(case)
    want = tx.ref_forward(lv, kind, g, x, w)
    try:
        _mode(F16)
        if cin % 64 and kind != "nin":
            rs = np.random.RandomState(1)
            gs = tx._geom(lv, "subm", 27)
            run_forward(lv, "subm", gs, torch.from_numpy(rs.randn(lv.n, 256).astype(np.float32)).cuda(), tx.grid_w(rs, 27, 256, 256))
        before = _counters()
        out, _ = run_forward(lv, kind, g, x, w)
        d = _delta(before)
        print(f"[fp16 exact] {tx._cid(case)} forward: {d}")
        tx.assert_exact(out, want, f"fp16 {tx._cid(case)} forward")
        tc = tx._expect_tc("bf16", kind, K, cout)
        assert d["tc"] == int(tc) and d["simt"] == int(not tc), d
        assert d["f16"] == int(_f16_forward(kind, K, cin, cout)), d
        total = d["f16"]
        if kind != "nin":
            before = _counters()
            d_in, dw = tx.run_backward(lv, kind, g, x, dy, w)
            d = _delta(before)
            print(f"[fp16 exact] {tx._cid(case)} backward: {d}")
            want_din, want_dw = tx.ref_backward(lv, kind, g, x, dy, w)
            tx.assert_exact(d_in, want_din, f"fp16 {tx._cid(case)} input gradient")
            tx.assert_exact(dw, want_dw, f"fp16 {tx._cid(case)} weight gradient")
            if tx._dw_tc_ok(cin, cout, K):
                assert d["f16"] >= 1, d
            total += d["f16"]
        assert total > 0
    finally:
        _mode(FP32)


@pytest.mark.parametrize("case,bias,addend", tx.EPI_CASES, ids=lambda v: tx._cid(v) if isinstance(v, tuple) else str(v))
def test_fused_epilogue_exact(case, bias, addend):
    """bias, the fused add and the 16-bit output copy, which must equal out.half()"""
    tx._tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, _ = tx._inputs(case, seed=1)
    rs = np.random.RandomState(cin + cout)
    b = tx.grid_w(rs, cout) if bias else None
    ad = tx.grid_w(rs, g["n_dst"], cout) if addend else None
    want = tx.ref_forward(lv, kind, g, x, w, b, ad)
    try:
        _mode(F16)
        before = _counters()
        out, o16 = run_forward(lv, kind, g, x, w, b, ad, want16=kind != "nin")
        d = _delta(before)
    finally:
        _mode(FP32)
    assert d["tc"] == 1 and d["f16"] == 1, d
    tx.assert_exact(out, want, f"fp16 {tx._cid(case)} epilogue")
    if o16 is not None:
        _same16(o16, out)


@pytest.mark.parametrize("c_lat", [32, 64, 128])
@pytest.mark.parametrize("kind,level", [("subm", "mini4"), ("deconv", "small"), ("subm", "big")])
def test_lateral_stage_and_epilogue_stats_exact(kind, level, c_lat):
    """out = conv(x) + y[row] @ W_lat in one launch, the lateral operand given as an fp16 copy, with the epilogue statistics"""
    tx._tc_or_skip()
    lv = tx._level(level)
    K = 27 if kind == "subm" else 8
    g = tx._geom(lv, kind, K)
    C0, n = 64, g["n_dst"]
    rs = np.random.RandomState(c_lat + K)
    density = 0.01 if level == "big" else 0.1
    x, w = tx.grid_x(rs, g["n_src"], C0, density), tx.grid_w(rs, K, C0, C0)
    y, wl = tx.grid_x(rs, n, c_lat, density), tx.grid_w(rs, c_lat, C0)
    want = tx.ref_forward(lv, kind, g, x, w) + y.double() @ wl.double()
    s1, s2 = want.sum(0), (want * want).sum(0)
    lib = _lib()
    try:
        _mode(F16)
        stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
        y16 = y.half()
        before = _counters()
        tx._check(lib.scn_fuse_next_lateral(tx._p(y), tx._p(y16), tx._p(wl), 0, c_lat, n))
        tx._check(lib.scn_fuse_next_stats(tx._p(stats)))
        out, _ = run_forward(lv, kind, g, x, w)
        took_l, took_s = C.c_int(), C.c_int()
        tx._check(lib.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
        d = _delta(before)
    finally:
        _mode(FP32)
    assert took_l.value == 1 and d["lateral"] == 1 and d["f16"] == 1, d
    tx.assert_exact(out, want, f"fp16 {kind} {level} lateral {c_lat}")
    if d["split"] == 0:
        assert took_s.value == 1 and d["stats"] == 1, d
        got1, got2 = tx._stats_sums(stats, C0)
        tx.assert_exact(got1, s1, "epilogue sum")
        tx.assert_exact(got2, s2, "epilogue sum of squares")


@pytest.mark.parametrize("case", tx.DW_CASES, ids=tx._cid)
def test_weight_gradient_exact(case):
    """d_W on conv_dw_tc with fp16 operands where dw_tc_ok takes the shape (one fp16 launch, the fp16 copy of d_out reused), on the
    CUDA-core k_dw elsewhere"""
    tx._tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, dy = tx._inputs(case, seed=2)
    _, want_dw = tx.ref_backward(lv, kind, g, x, dy, w)
    try:
        _mode(F16)
        before = _counters()
        _, dw = tx.run_backward(lv, kind, g, x, dy, w, want_din=kind != "subm")
        d = _delta(before)
    finally:
        _mode(FP32)
    print(f"[fp16 dw] {tx._cid(case)}: {d}")
    tc = tx._dw_tc_ok(cin, cout, K)
    launches = d["atomic"] - d["split"]
    assert (launches == 1) == tc, d
    if tc:
        assert d["f16"] >= 1, d
        if cin % 32 == 0:
            assert d["reused"] >= 1, d
    tx.assert_exact(dw, want_dw, f"fp16 {tx._cid(case)} weight gradient")


def test_wide_plan_chunks_exact():
    """5^3 submanifold (125 offsets: two chunked launches) forward and backward, bit for bit"""
    tx._tc_or_skip()
    lv = tx._level("small")
    g = dict(a=lv.full, b=lv.full, f=[5, 5, 5], s=[1, 1, 1], n_src=lv.n, n_dst=lv.n, key=("subm", (5, 5, 5)))
    rs = np.random.RandomState(125)
    for cin, cout in ((64, 64), (32, 32)):
        x, w, dy = tx.grid_x(rs, lv.n, cin, 0.2), tx.grid_w(rs, 125, cin, cout), tx.grid_w(rs, lv.n, cout)
        want = tx.ref_forward(lv, "subm", g, x, w)
        want_din, want_dw = tx.ref_backward(lv, "subm", g, x, dy, w)
        try:
            _mode(F16)
            before = _counters()
            out, o16 = run_forward(lv, "subm", g, x, w, want16=True)
            d = _delta(before)
            d_in, dw = tx.run_backward(lv, "subm", g, x, dy, w)
        finally:
            _mode(FP32)
        assert d["chunk"] == 2 and d["f16"] == 2, d
        tx.assert_exact(out, want, f"5^3 {cin}")
        _same16(o16, out)
        tx.assert_exact(d_in, want_din, f"5^3 {cin} input gradient")
        tx.assert_exact(dw, want_dw, f"5^3 {cin} weight gradient")


def test_deterministic_mode_exact():
    """split-offset partials (k_split_sum with the fp16 copy), a large level and the weight gradient's ordered parts, with and
    without torch.use_deterministic_algorithms(True): equal to the reference bit for bit"""
    tx._tc_or_skip()
    cases = [("subm", "small", 27, 64, 64), ("subm", "big", 27, 32, 32), ("deconv", "small", 8, 128, 64)]
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        _mode(F16)
        for case in cases:
            kind = case[0]
            lv, g, x, w, dy = tx._inputs(case, seed=3)
            want = tx.ref_forward(lv, kind, g, x, w)
            want_din, want_dw = tx.ref_backward(lv, kind, g, x, dy, w)
            for flag in (False, True):
                torch.use_deterministic_algorithms(flag)
                before = _counters()
                out, o16 = run_forward(lv, kind, g, x, w, want16=True)
                d_in, dw = tx.run_backward(lv, kind, g, x, dy, w)
                d = _delta(before)
                torch.use_deterministic_algorithms(on, warn_only=warn)
                tag = f"{'deterministic' if flag else 'default'} {tx._cid(case)}"
                assert d["f16"] >= 2, (tag, d)
                if flag:
                    assert d["atomic"] == 0, (tag, d)
                tx.assert_exact(out, want, tag + " forward")
                _same16(o16, out)
                tx.assert_exact(d_in, want_din, tag + " input gradient")
                tx.assert_exact(dw, want_dw, tag + " weight gradient")
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        _mode(FP32)


# ------------------------------------------------------------------ 3. operand convention
def _nin_probe(x, w):
    lv = tx._level("rows1")  # (dense rows: no Metadata involved)
    g = dict(n_src=x.shape[0], n_dst=x.shape[0])
    try:
        _mode(F16)
        before = _counters()
        out, _ = run_forward(lv, "nin", g, x, w)
        d = _delta(before)
    finally:
        _mode(FP32)
    assert d["tc"] == 1 and d["f16"] == 1, d
    return out


@pytest.mark.parametrize("cin", [64, 9, 20])
def test_operand_rounding_convention(cin):
    """One active channel per row, so every output is ONE product of two rounded operands, exact in fp32.  fp16 keeps 10 of fp32's
    23 mantissa bits: in the normal range its rounding is the TF32 rounding of the same value, so tx._tf32 names the candidates.
    Activations (through k_to_16 for 64 channels, the zero-padding copy for 9 and 20) and weights round to nearest even."""
    tx._tc_or_skip()
    n, cout = 128, 32
    rs = np.random.RandomState(cin + 16)
    ch = torch.from_numpy(np.arange(n) % cin).cuda()
    found = {}
    for operand in ("act", "weight"):
        a = tx._probe_values(rs, n, 13) if operand == "act" else torch.from_numpy(rs.choice([-2.0, -1.0, 1.0, 2.0], n).astype(np.float32)).cuda()
        w = (tx._probe_values(rs, cin * cout, 13) if operand == "weight" else tx._probe_values(rs, cin * cout, 13).half().float()).view(cin, cout)
        x = torch.zeros(n, cin, device="cuda")
        x[torch.arange(n, device="cuda"), ch] = a
        out = _nin_probe(x, w)
        match = []
        for how in ("trunc", "rna", "rne"):
            ra, rw = (tx._tf32(a, how), w) if operand == "act" else (a, tx._tf32(w, how))
            if torch.equal(out.double(), ra.double()[:, None] * rw.double()[ch]):
                match.append(how)
        found[operand] = match
        if operand == "act":
            assert torch.equal(tx._tf32(a, "rne"), a.half().float())  # (the rne candidate is torch's .half())
    print(f"[fp16 rounding] Cin={cin}: activations {found['act']}, weights {found['weight']}")
    assert found["act"] == ["rne"] and found["weight"] == ["rne"], found


def test_subnormal_and_overflow():
    """2^-20 (an fp16 subnormal) survives as an activation and as a weight; an activation of 7e4 (> 65504) becomes inf and the
    inf reaches the output: no flush to zero, no saturation"""
    tx._tc_or_skip()
    n, cin, cout = 128, 64, 32
    x = torch.zeros(n, cin, device="cuda")
    x[:, 0] = 1.0
    x[0, 0], x[1, 0], x[2, 0], x[3, 0] = 2.0 ** -20, -(2.0 ** -20), 7e4, -7e4
    w = torch.zeros(cin, cout, device="cuda")
    w[0] = 1.0
    w[0, 1] = 2.0 ** -20
    w[0, 2] = 0.5
    out = _nin_probe(x, w)
    assert float(out[0, 0]) == 2.0 ** -20 and float(out[1, 0]) == -(2.0 ** -20), out[:2, :3]
    assert float(out[4, 1]) == 2.0 ** -20, out[4, :3]  # the weight
    assert float(out[4, 0]) == 1.0
    assert torch.isinf(out[2, 0]) and float(out[2, 0]) > 0 and torch.isinf(out[3, 0]) and float(out[3, 0]) < 0, out[2:4, :3]
    assert torch.isinf(out[2, 2]), out[2, :3]
    assert torch.isfinite(out[4:]).all()


# ------------------------------------------------------------------ 4. per layer on random data
LAYER_CASES = [  # (kind, level, K, cin, cout)
    ("subm", "mini4", 27, 64, 64), ("subm", "big", 27, 128, 128), ("subm", "small", 1, 64, 128), ("conv", "small", 8, 64, 128),
    ("deconv", "small", 8, 128, 64), ("conv", "small", 16, 64, 64), ("nin", "mini4", 1, 192, 64), ("subm", "big", 27, 32, 32),
    ("subm", "mini4", 27, 9, 32),
]


@pytest.mark.parametrize("case", LAYER_CASES, ids=tx._cid)
def test_layer_random_data(case):
    """N(0, 1) activations, He-scaled weights: fp16 within tf32's per-layer bounds of the exact result, and no less accurate than
    bf16 on the same data.  Covers submanifold 3^3 and 1^3, strided, deconvolution, z-collapse, NetworkInNetwork, packed 32-channel
    rows and the 9 -> 32 input convolution (16-channel packed rows)."""
    tx._tc_or_skip()
    kind, level, K, cin, cout = case
    lv = tx._level(level)
    g = tx._geom(lv, kind, K)
    rs = np.random.RandomState(cin * 7 + cout + K)
    x = torch.from_numpy(rs.randn(g["n_src"], cin).astype(np.float32)).cuda()
    shape = (cin, cout) if kind == "nin" else (K, cin, cout)
    w = torch.from_numpy((rs.randn(*shape) * (2.0 / (cin * K)) ** 0.5).astype(np.float32)).cuda()
    ref = tx.ref_forward(lv, kind, g, x, w)
    scale = max(1.0, float(ref.abs().max()))
    errs = {}
    for mode in (F16, BF16):
        try:
            _mode(mode)
            before = _counters()
            out, _ = run_forward(lv, kind, g, x, w)
            d = _delta(before)
        finally:
            _mode(FP32)
        assert d["f16"] == int(mode == F16), d
        errs[mode] = float((out.double() - ref).abs().max()) / scale
        if mode == F16:
            np.testing.assert_allclose(out.cpu().numpy(), ref.cpu().numpy(), rtol=LAYER_RTOL, atol=LAYER_ATOL * scale)
    print(f"[fp16 layer] {tx._cid(case)}: max|d| / max|ref| fp16 {errs[F16]:.2e}, bf16 {errs[BF16]:.2e}")
    assert errs[F16] <= errs[BF16], errs


def test_accumulation_error_bound():
    """tx.test_accumulation_error_bound for fp16 mode: against the fp64 sum of the operands as the kernel rounds them (fp16 where
    the layer has 16-bit operands, TF32 otherwise), what is left is the fp32 accumulation, within bf16's tau"""
    tx._tc_or_skip()
    worst = 0.0
    for case in tx.BOUND_CASES:
        kind, level, K, cin, cout = case
        lv = tx._level(level)
        g = tx._geom(lv, kind, K)
        rs = np.random.RandomState(cin + cout)
        x = torch.from_numpy(rs.randn(g["n_src"], cin).astype(np.float32)).cuda()
        w = torch.from_numpy((rs.randn(*((cin, cout) if kind == "nin" else (K, cin, cout))) * (1 / (cin * K)) ** 0.5).astype(np.float32)).cuda()
        try:
            _mode(F16)
            out, _ = run_forward(lv, kind, g, x, w)
        finally:
            _mode(FP32)
        if _f16_forward(kind, K, cin, cout):
            terms = [(x.half().float(), w.half().float())]
        else:
            terms = [(tx._tf32(x, tx.TF32_ACT), tx._tf32(w, "rna"))]
        ref_r = sum(tx.ref_forward(lv, kind, g, a, b) for a, b in terms)
        S = sum(tx.ref_forward(lv, kind, g, a.abs(), b.abs()) for a, b in terms)
        ratio = float(((out.double() - ref_r).abs() / S.clamp_min(1e-300)).max())
        print(f"[fp16 bound] {tx._cid(case)}: {ratio:.3e} ({ratio * 2 ** 24:.2f} x 2^-24)")
        worst = max(worst, ratio)
    assert worst <= tx.TAU["bf16"], (worst, tx.TAU["bf16"])


# ------------------------------------------------------------------ 5. end to end
def _fpn(scn, cfg, seed=1, train=False):
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=seed))
    return net.cuda().train() if train else net.cuda().eval()


def _e2e_err(rpn, roi, g):
    worst = 0.0
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        assert len(maps) == int(g[f"n_{tag}"])
        for i, m in enumerate(maps):
            assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
            ref = g[f"{tag}{i}_features"]
            err = float(np.abs(m.features.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max()))
            worst = max(worst, err)
    return worst


@pytest.mark.parametrize("name,cfgname,bld", [("mini4", "mini4", MINI4_BLD), ("sw4c_mid", "sw4c", MID_BLD)])
def test_fpn_forward_vs_reference_golden(name, cfgname, bld):
    """Layer by layer (recording), two replays, and a replay on a prefetched Metadata, each within E2E of the reference's outputs"""
    scn = _scn()
    cfg = fpn_util.mini4_config() if cfgname == "mini4" else scn.sw4c_fpn432_config()
    g = np.load(os.path.join(GOLD, f"fpn_{name}.npz"))
    coords = synthetic.building_coords(**bld)
    c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()
    errs = []
    try:
        scn.set_math_mode("fp16")
        net = _fpn(scn, cfg)
        with torch.no_grad():
            for rep in range(3):
                before = _counters()
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])  # records, then replays
                torch.cuda.synchronize()
                d = _delta(before)
                assert d["f16"] > 0, d
                assert scn.forward_pass_multiplyAdd_count == float(g["macs"])
                errs.append(_e2e_err(rpn, roi, g))
                if rep == 0:
                    assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
            cd = c.cuda()
            torch.cuda.synchronize()
            assert net.prefetch(cd)
            rpn, roi = net([cd, f])
            errs.append(_e2e_err(rpn, roi, g))
    finally:
        scn.set_math_mode("fp32")
    print(f"[fp16 e2e] {name}: max|d| / max(1, max|ref|) per pass (recording, replay, replay, prefetched) " + ", ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= E2E, errs


# ------------------------------------------------------------------ 6. training
def _train_step(scn, net, coords, scale=1.0):
    rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
    terms = [(m.features ** 2).mean() for m in rpn + roi]
    loss = sum(terms)
    (loss * scale).backward()
    torch.cuda.synchronize()
    return terms, loss


@pytest.mark.parametrize("replay", [False, True])
def test_training_step_vs_reference_autograd(replay):
    """The mini4 training step (tests/golden/fpn_mini4_train.npz) against the reference's autograd; then the same step at loss scale
    2^12, its gradients divided by the scale, agrees with the unscaled one (worst element within 1.5e-1 of max|grad|, measured 6.1e-2:
    the unscaled step loses the output gradients below fp16's normal range, 2^-14, that the scaled one keeps; relative rms of the
    whole gradient vector within 2e-2, measured <= 4.8e-3; cosine at least 0.9999, measured >= 0.99998).  Bounds against the reference: tf32's relative rms, cosine and loss bounds of
    test_gpu_pins.py; on the worst element bf16's, 5e-1.  Measured on an NVIDIA B200 (1000 W): rms <= 5.3e-2, worst element 3.6e-1,
    in the weight gradient of the deepest level (m_downs.3), where train-mode BatchNorm over a few dozen rows amplifies the rounding
    of the fp16 operands of the weight-gradient kernel and of the output-gradient copies (tf32 mode runs those weight gradients on
    the exact CUDA-core kernel)."""
    scn = _scn()
    g = np.load(os.path.join(GOLD, "fpn_mini4_train.npz"))
    tol_max, tol_rms, tol_cos, tol = 5e-1, 8e-2, 0.995, 3e-2
    coords = synthetic.building_coords(**MINI4_BLD)
    cfg = dict(fpn_util.mini4_config(), track_running_stats=True)
    try:
        scn.set_math_mode("fp16")
        net = _fpn(scn, cfg, train=True)
        if replay:
            _train_step(scn, net, coords)
            assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
            net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
            net.zero_grad(set_to_none=True)
        before = _counters()
        terms, loss = _train_step(scn, net, coords)
        d = _delta(before)
        grads = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net.zero_grad(set_to_none=True)
        _train_step(scn, net, coords, scale=2.0 ** 12)
        scaled = {k: p.grad / 2.0 ** 12 for k, p in net.named_parameters() if p.grad is not None}
    finally:
        scn.set_math_mode("fp32")
    assert d["f16"] > 0 and d["train_replay"] == (1 if replay else 0), d
    np.testing.assert_allclose(np.array([float(t.detach()) for t in terms]), g["map_mean_sq"], rtol=tol)
    assert abs(float(loss) - float(g["loss"])) <= tol * float(g["loss"])
    want_keys = {k[5:] for k in g.files if k.startswith("grad:")}
    assert set(grads) == want_keys
    worst, worst_scaled = 0.0, 0.0
    for k in want_keys:
        ref = g["grad:" + k].astype(np.float64)
        dd = grads[k].cpu().numpy().astype(np.float64) - ref
        err = float(np.abs(dd).max() / max(1e-6, np.abs(ref).max()))
        rms = float(np.sqrt((dd * dd).mean()) / max(1e-12, np.sqrt((ref * ref).mean())))
        worst = max(worst, err)
        assert err < tol_max and rms < tol_rms, (k, err, rms)
        a, b = grads[k].double(), scaled[k].double()
        worst_scaled = max(worst_scaled, float((a - b).abs().max()) / max(1e-6, float(a.abs().max())))
    keys = sorted(want_keys)
    a = np.concatenate([grads[k].cpu().numpy().ravel() for k in keys]).astype(np.float64)
    b = np.concatenate([g["grad:" + k].ravel() for k in keys]).astype(np.float64)
    cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)))
    s_ = np.concatenate([scaled[k].cpu().numpy().ravel() for k in keys]).astype(np.float64)
    rms_scaled = float(np.linalg.norm(s_ - a) / np.linalg.norm(a))
    cos_scaled = float(a @ s_ / (np.linalg.norm(a) * np.linalg.norm(s_)))
    print(f"[fp16] training step (replay={replay}): worst gradient error {worst:.3e} of max|grad|, cosine {cos:.6f}; "
          f"loss scale 2^12 vs unscaled: worst {worst_scaled:.3e} of max|grad|, rel. rms {rms_scaled:.3e}, cosine {cos_scaled:.8f}")
    assert cos >= tol_cos, cos
    assert worst_scaled <= 1.5e-1 and rms_scaled <= 2e-2 and cos_scaled >= 0.9999, (worst_scaled, rms_scaled, cos_scaled)


def test_grad_scaler_skips_overflowing_step():
    """torch.amp.GradScaler with an initial scale of 2^40: the scaled output gradients exceed fp16's range, become inf in the fp16
    operand copies and reach the parameter gradients; scaler.step skips the update and update() lowers the scale."""
    scn = _scn()
    coords = synthetic.building_coords(**MINI4_BLD)
    try:
        scn.set_math_mode("fp16")
        net = _fpn(scn, dict(fpn_util.mini4_config(), track_running_stats=True), train=True)
        opt = torch.optim.SGD(net.parameters(), lr=0.1)
        scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40)
        params = {k: p.detach().clone() for k, p in net.named_parameters()}
        rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()])
        loss = sum((m.features ** 2).mean() for m in rpn + roi)
        scaler.scale(loss).backward()
        nonfinite = sum(int(not torch.isfinite(p.grad).all()) for p in net.parameters() if p.grad is not None)
        scaler.step(opt)
        scaler.update()
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert nonfinite > 0
    for k, p in net.named_parameters():
        assert torch.equal(p.detach(), params[k]), k
    assert scaler.get_scale() < 2.0 ** 40


# ------------------------------------------------------------------ 7. switching between bf16 and fp16
def test_switch_between_layers_and_forwards():
    """bf16 -> fp16 -> bf16 between the layers of one layer-by-layer run (BatchNorm outputs carry 16-bit shadows) and between
    whole forwards: every result equals the same step of single-mode runs, so no shadow or weight image of the other format was
    consumed"""
    scn = _scn()
    from detection_3d_b200.sparseconvnet import native
    from gpu_adapter import GpuMetadata
    coords, full = synthetic.building_coords(**MINI4_BLD), [64, 64, 32]
    G = GpuMetadata()
    n = G.input_layer(full, coords, 0, 4)
    rs = np.random.RandomState(5)
    x = torch.from_numpy(rs.randn(n, 64).astype(np.float32)).cuda()
    ws = [torch.from_numpy((rs.randn(27, 1, 64, 64) * (2 / (64 * 27)) ** 0.5).astype(np.float32)).cuda() for _ in range(3)]
    L = torch.LongTensor

    def layer(h, w):
        y, sm, si = torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        native.BatchNormalization_updateOutput(h, y, sm, si, torch.Tensor(), torch.Tensor(), torch.Tensor(), torch.Tensor(), 1e-4, 0.9,
                                               False, 0.0, instance_stats=True)
        out = torch.empty(0, device="cuda")
        native.SubmanifoldConvolution_updateOutput(L(full), L([3, 3, 3]), G.m, y, out, w, torch.Tensor())
        return out

    def run(modes):
        h, outs = x, []
        for m, w in zip(modes, ws):
            scn.set_math_mode(m)
            h = layer(h, w)
            outs.append(h.clone())
        torch.cuda.synchronize()
        return outs
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)  # (fixed summation order of the BatchNorm statistics: bitwise comparisons)
    try:
        single = {m: run([m] * 3) for m in ("bf16", "fp16")}
        mixed = run(["bf16", "fp16", "bf16"])
        again = {m: run([m] * 3) for m in ("fp16", "bf16")}
        before = _counters()
        scn.set_math_mode("fp16")
        h1 = layer(x, ws[0])
        d = _delta(before)
    except BaseException:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        scn.set_math_mode("fp32")
        raise
    assert d["f16"] == 1, d
    for m in ("bf16", "fp16"):  # whole runs, one mode each, after the other mode's run: the same bits
        for a, b in zip(single[m], again[m]):
            assert torch.equal(a, b), m
    assert torch.equal(mixed[0], single["bf16"][0])
    assert torch.equal(h1, single["fp16"][0])
    assert not torch.equal(single["bf16"][0], single["fp16"][0])
    # layer 2 of the mixed run read an fp32 input whose bf16 shadow it must ignore: it equals fp16 on the bf16 layer-1 output
    try:
        scn.set_math_mode("fp16")
        ref2 = layer(mixed[0], ws[1])
        scn.set_math_mode("bf16")
        ref3 = layer(mixed[1], ws[2])
        torch.cuda.synchronize()
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        scn.set_math_mode("fp32")
    assert torch.equal(mixed[1], ref2) and torch.equal(mixed[2], ref3)


def test_switch_between_recorded_forwards():
    """Forwards of one network in bf16, fp16, bf16, fp16 (two per switch) equal those of fresh single-mode networks.  FPN_Net keeps
    the program it recorded in its first mode (bf16) and runs the forwards of any other mode layer by layer: the bf16 forwards after
    the first are replays and equal a fresh bf16 network's replay, the fp16 ones equal a fresh fp16 network's first (layer-by-layer)
    forward -- so neither path consumed a weight image or shadow the other mode left behind."""
    scn = _scn()
    coords = synthetic.building_coords(**MINI4_BLD)
    c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()
    cfg = fpn_util.mini4_config()

    def fwd(net):
        with torch.no_grad():
            rpn, roi = net([c, f])
        torch.cuda.synchronize()
        return [m.features.clone() for m in rpn + roi]

    def equal(a, b, what):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            assert torch.equal(x, y), (what, i, float((x - y).abs().max()))
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(True)  # (small levels split filter offsets: bitwise comparisons need the fixed order)
        net = _fpn(scn, cfg)
        seq = []
        for m in ("bf16", "fp16", "bf16", "fp16"):
            scn.set_math_mode(m)
            before = _counters()
            seq.append((m, fwd(net), fwd(net), _delta(before)))
        fresh = {}
        for m in ("bf16", "fp16"):
            scn.set_math_mode(m)
            other = _fpn(scn, cfg)
            fresh[m] = (fwd(other), fwd(other))  # layer by layer (records), replay
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        scn.set_math_mode("fp32")
    for i, (m, a, b, d) in enumerate(seq):
        assert (d["f16"] > 0) == (m == "fp16"), (i, m, d)
        if m == "bf16":
            equal(a, fresh[m][0] if i == 0 else fresh[m][1], f"bf16 forward {i}, first")
            equal(b, fresh[m][1], f"bf16 forward {i}, second")
        else:
            equal(a, fresh[m][0], f"fp16 forward {i}, first")
            equal(b, fresh[m][0], f"fp16 forward {i}, second")


# ------------------------------------------------------------------ 8. deterministic mode, whole network
def test_deterministic_network():
    """Under torch.use_deterministic_algorithms(True), fp16 mode: recording forwards of two fresh networks, two replays and two
    replayed training steps are bitwise equal, and no launch accumulated floats with atomics"""
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
        sum((m.features ** 2).mean() for m in rpn + roi).backward()
        torch.cuda.synchronize()
        return ([p.grad.clone() for _, p in sorted(net.named_parameters()) if p.grad is not None] + [x.grad.clone()]
                + [b.clone() for _, b in sorted(net.named_buffers())])

    def equal(a, b):
        assert len(a) == len(b)
        for i, (u, v) in enumerate(zip(a, b)):
            assert u.shape == v.shape and torch.equal(u, v), i
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        scn.set_math_mode("fp16")
        before = _counters()
        a, b = _fpn(scn, fpn_util.mini4_config()), _fpn(scn, fpn_util.mini4_config())
        equal(forward(a), forward(b))
        equal(forward(a), forward(a))
        tnet = _fpn(scn, dict(fpn_util.mini4_config(), track_running_stats=True), train=True)
        state = {k: v.clone() for k, v in tnet.state_dict().items()}
        step(tnet, state)
        assert tnet.__dict__.get("_program_train") is not None, tnet.__dict__.get("_program_train_error")
        equal(step(tnet, state), step(tnet, state))
        d = _delta(before)
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        scn.set_math_mode("fp32")
    assert d["atomic"] == 0 and d["f16"] > 0, d
