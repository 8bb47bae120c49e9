"""The tensor-core convolution kernels (csrc/conv_tc.cu: conv_plan_tc, conv_dw_tc, conv_dw_plan_tc) against a plain float64
gather-GEMM over the oracle's rule pairs, bit for bit.

Exact grid: activations in {-1, 0, 1}; weights, output gradients, bias and addend in {k/8 : |k| <= 3}.  Every product and every
partial sum is then a multiple of 1/8 far below 2^21: exactly representable in fp32, and the operands are exact in TF32 and bf16
(tf32x3 splits them with lo = 0).  Each convolution has exactly one correct fp32 result, whatever the summation order, the split of
the filter offsets, the atomics or the schedule, and every path must return it (DESIGN.md section 7).  Inputs are the leading rows of
buffers with a NaN tail, outputs land in buffers with a sentinel tail that must stay untouched.

Also here: the rounding convention of each operand (single-product probes), an accumulation-error bound per math mode on random
data, and every launcher knob of conv_tc.cu in a subprocess of its own (the knobs are read once per process).

Run time on a B200: about 2 minutes."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from detection_3d_b200 import synthetic
from oracle import scn_oracle as so

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = {"fp32": 0, "tf32": 1, "bf16": 2, "tf32x3": 3}
TC_MODES = ("tf32", "bf16", "tf32x3")
CNT = dict(lateral=3, stats=4, tc=7, split=9, simt=10, reused=12, dw_plan=13, atomic=14, x3=15)
SENT = -3 * 2.0 ** -10  # sentinel of output tails: exact in fp32 and bf16, not a multiple of 1/8 (no grid result)
GUARD = 131     # rows of NaN / sentinel beyond the last real row
# How the tensor core reads raw fp32 activation rows in tf32 mode (the weights are converted with cvt.rna by k_prep_wimg):
# measured by test_operand_rounding_convention on B200
TF32_ACT = "trunc"
# max over outputs of |got - ref_r| / sum|products|, ref_r = fp64 sum of the operands rounded as the kernel rounds them.
# tau = 4x the maximum test_accumulation_error_bound measured on an NVIDIA B200 (1000 W): fp32 4.7e-7 (7.9 x 2^-24), tf32 9.5e-7
# (16 x 2^-24), bf16 4.9e-7 (8.1 x 2^-24), tf32x3 2.6e-6 (43 x 2^-24: three MMAs per K step into one accumulator).  DESIGN.md section 7.
TAU = {"fp32": 4 * 4.72e-7, "tf32": 4 * 9.52e-7, "bf16": 4 * 4.86e-7, "tf32x3": 4 * 2.59e-6}


def _lib():
    from detection_3d_b200._lib import lib
    return lib()


def _check(status):
    from detection_3d_b200._lib import check
    check(status)


def _l3(v):
    from detection_3d_b200._lib import l3
    return l3(v)


def _tc_or_skip():
    if not _lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")


def _counters():
    return {k: _lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _set_mode(mode):
    _check(_lib().scn_set_math_mode(MODES[mode]))


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


# ------------------------------------------------------------------ levels
def _coords(name):
    """(coords [n, 4] = x, y, z, batch, spatial size) of a named level"""
    if name == "small":
        return synthetic.small_building(40, 36, 12, 3, seed=4), [64, 64, 32]
    if name == "mini4":  # 111 tiles: more items than the split limit, fewer tiles than SMs
        return synthetic.building_coords(nx=60, ny=56, nz=24, n_walls=3, seed=3), [64, 64, 32]
    if name == "big":    # 277k rows: many super-tiles, ragged last tile
        return synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5), [2048, 2048, 512]
    if name == "lines":  # 10 lines of 4000 sites 2 apart in y, 3 sites between them: 3 long rule lists, 6 lists of 1-3 rules, 18 empty
        x = np.arange(4000)
        c = [np.stack([x, np.full_like(x, 2 * j), np.zeros_like(x)], 1) for j in range(10)]
        c.append(np.array([[10, 1, 0], [1000, 1, 0], [3000, 1, 0]]))
        c = np.concatenate(c)
        return np.concatenate([c, np.zeros((len(c), 1), c.dtype)], 1), [4096, 32, 4]
    assert name.startswith("rows")  # n sites of a 6 x 6 x 6 block: one ragged tile (1 ... 129 rows)
    n = int(name[4:])
    g = np.stack(np.meshgrid(np.arange(6), np.arange(6), np.arange(6), indexing="ij"), -1).reshape(-1, 3)
    g = g[np.random.RandomState(n).permutation(len(g))[:n]]
    return np.concatenate([g, np.zeros((n, 1), g.dtype)], 1), [16, 16, 16]


class _Level:
    def __init__(self, name):
        from gpu_adapter import GpuMetadata
        self.coords, self.full = _coords(name)
        self.G = GpuMetadata()
        self.n = self.G.input_layer(self.full, self.coords, 0, 4)
        self._O, self._rules, self._made, self._o_made = None, {}, [], set()

    @property
    def O(self):  # the CPU oracle, for the rule pairs of the references (subprocesses never need it)
        if self._O is None:
            self._O = so.OracleMetadata()
            assert self._O.input_layer(self.full, self.coords, 0, 4) == self.n
        return self._O

    def nactive(self, sz):
        return int(self.G.nactive(sz))

    def make_conv(self, a, b, f, s):  # the GPU-side rulebook a -> b (a deconvolution b -> a looks it up)
        key = tuple(map(tuple, (a, b, f, s)))
        if key not in self._made:
            self.G.conv_rules(a, b, f, s)
            self._made.append(key)

    def rules(self, key):
        """per filter offset, (in row, out row) pairs of the convolution `key` as int64 device tensors"""
        for k in self._made:  # the oracle builds the coarser grids in the same order
            if k not in self._o_made:
                self.O.conv_rules(*[list(v) for v in k])
                self._o_made.add(k)
        if key not in self._rules:
            r = self.O.submanifold_rules(self.full, list(key[1])) if key[0] == "subm" else self.O.conv_rules(*[list(v) for v in key[1:]])
            self._rules[key] = [torch.from_numpy(np.ascontiguousarray(x, np.int64)).cuda() for x in r]
        return self._rules[key]


_LEVELS = {}


def _level(name):
    if name not in _LEVELS:
        _LEVELS[name] = _Level(name)
    return _LEVELS[name]


def _geom(lv, kind, K):
    """spatial sizes, filter and stride of a layer; `a` is the finer grid, the layer reads rows of `src` and writes rows of `dst`"""
    full = lv.full
    half = [v // 2 for v in full]
    if kind in ("subm", "nin"):
        f = {1: 1, 27: 3}[K]
        return dict(a=full, b=full, f=[f] * 3, s=[1, 1, 1], n_src=lv.n, n_dst=lv.n, key=("subm", (f, f, f)))
    if K == 8:
        a, b, f, s = full, half, [2, 2, 2], [2, 2, 2]
    elif K == 64:  # f = 4^3, stride 2: the last filter offset uses tile-mask bit 63
        a, b, f, s = full, [(v - 4) // 2 + 1 for v in full], [4, 4, 4], [2, 2, 2]
    else:          # K = 16: z-collapse of the coarse level
        assert K == 16
        lv.make_conv(full, half, [2, 2, 2], [2, 2, 2])
        a, b, f, s = half, [half[0], half[1], 1], [1, 1, half[2]], [1, 1, 1]
    lv.make_conv(a, b, f, s)
    na, nb = lv.nactive(a), lv.nactive(b)
    g = dict(a=a, b=b, f=f, s=s, key=("conv", tuple(a), tuple(b), tuple(f), tuple(s)))
    return dict(g, n_src=na, n_dst=nb) if kind == "conv" else dict(g, n_src=nb, n_dst=na)


# ------------------------------------------------------------------ fp64 reference (plain gather-GEMM, nothing from the library)
def _pairs(lv, kind, g, k):
    r = lv.rules(g["key"])[k]
    return (r[:, 1], r[:, 0]) if kind == "deconv" else (r[:, 0], r[:, 1])


def ref_forward(lv, kind, g, x, w, bias=None, addend=None):
    """out[o] += x[i] @ W[k] over the (i, o) pairs of offset k (reversed for a deconvolution), in float64"""
    x, w = x.double(), w.double()
    if kind == "nin":
        out = x @ w
    else:
        out = torch.zeros(g["n_dst"], w.shape[-1], dtype=torch.float64, device=x.device)
        for k in range(w.shape[0]):
            i, o = _pairs(lv, kind, g, k)
            if len(i):
                out.index_add_(0, o, x[i] @ w[k])
    if bias is not None:
        out += bias.double()
    if addend is not None:
        out += addend.double()
    return out


def ref_backward(lv, kind, g, x, dy, w):
    """(d_in, d_W): d_in[i] += dy[o] @ W[k]^T and dW[k] = sum x[i]^T dy[o] over the pairs, in float64"""
    x, dy, w = x.double(), dy.double(), w.double()
    d_in = torch.zeros_like(x)
    dw = torch.zeros_like(w)
    for k in range(w.shape[0]):
        i, o = _pairs(lv, kind, g, k)
        if len(i):
            d_in.index_add_(0, i, dy[o] @ w[k].t())
            dw[k] = x[i].t() @ dy[o]
    return d_in, dw


# ------------------------------------------------------------------ inputs on the exact grid
def grid_x(rs, n, c, density=2 / 3):
    v = rs.choice([-1.0, 1.0], (n, c)) * (rs.rand(n, c) < density)
    return torch.from_numpy(v.astype(np.float32)).cuda()


def grid_w(rs, *shape):
    return torch.from_numpy((rs.randint(-3, 4, shape) / 8).astype(np.float32)).cuda()


def _guarded(x, fill):
    buf = torch.full((x.shape[0] + GUARD,) + tuple(x.shape[1:]), fill, dtype=x.dtype, device="cuda")
    buf[:x.shape[0]] = x
    return buf


def _tail_untouched(buf, n, what):
    tail = buf[n:].float()
    assert bool((tail == SENT).all()), f"{what}: {int((tail != SENT).sum())} elements beyond the last row were written"


def run_forward(lv, kind, g, x, w, bias=None, addend=None, want16=False):
    """one forward call through the C ABI into guarded buffers -> (out fp32, out bf16 or None)"""
    lib = _lib()
    n_in, cin = x.shape
    cout, n = w.shape[-1], g["n_dst"]
    xb = _guarded(x, float("nan"))
    ob = torch.full((n + GUARD, cout), SENT, device="cuda")
    o16 = torch.full((n + GUARD, cout), SENT, dtype=torch.bfloat16, device="cuda") if want16 else None
    macs = C.c_double()
    h = lv.G.m._h
    if kind == "nin":
        assert addend is None and not want16
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _check(lib.scn_network_in_network_forward(_p(xb), _p(ob), _p(w), _p(bias), n_in, cin, cout, C.byref(macs), stream, None, 0))
    else:
        args = (_p(xb), _p(ob), _p(w), _p(bias), cin, cout, C.byref(macs), None, 0, _p(addend), _p(o16))
        if kind == "subm":
            _check(lib.scn_submanifold_convolution_forward(h, _l3(g["a"]), _l3(g["f"]), *args))
        elif kind == "conv":
            _check(lib.scn_convolution_forward(h, _l3(g["a"]), _l3(g["b"]), _l3(g["f"]), _l3(g["s"]), *args))
        else:
            _check(lib.scn_deconvolution_forward(h, _l3(g["b"]), _l3(g["a"]), _l3(g["f"]), _l3(g["s"]), *args))
    torch.cuda.synchronize()
    _tail_untouched(ob, n, "forward output")
    if want16:
        _tail_untouched(o16, n, "bf16 output copy")
    return ob[:n], (o16[:n] if want16 else None)


def run_backward(lv, kind, g, x, dy, w, want_din=True):
    """one backward call through the C ABI -> (d_in or None, d_W); d_bias is not requested"""
    lib = _lib()
    cin, cout, K = x.shape[1], dy.shape[1], w.shape[0]
    xb, dyb = _guarded(x, float("nan")), _guarded(dy, float("nan"))
    din = torch.full((x.shape[0] + GUARD, cin), SENT, device="cuda") if want_din else None
    dw = torch.full((K * cin * cout + 64,), SENT, device="cuda")
    h = lv.G.m._h
    args = (_p(xb), _p(din), _p(dyb), _p(w), _p(dw), None, cin, cout)
    if kind == "subm":
        _check(lib.scn_submanifold_convolution_backward(h, _l3(g["a"]), _l3(g["f"]), *args))
    elif kind == "conv":
        _check(lib.scn_convolution_backward(h, _l3(g["a"]), _l3(g["b"]), _l3(g["f"]), _l3(g["s"]), *args))
    else:
        _check(lib.scn_deconvolution_backward(h, _l3(g["b"]), _l3(g["a"]), _l3(g["f"]), _l3(g["s"]), *args))
    torch.cuda.synchronize()
    _tail_untouched(dw, K * cin * cout, "weight gradient")
    if want_din:
        _tail_untouched(din, x.shape[0], "input gradient")
    return (din[:x.shape[0]] if want_din else None), dw[:K * cin * cout].view(K, cin, cout)


def assert_exact(got, want, what):
    """bitwise equality of an fp32 result with the (exactly representable) fp64 reference"""
    assert got.shape == want.shape, (what, tuple(got.shape), tuple(want.shape))
    assert torch.equal(want.float().double(), want), f"{what}: the reference is not exactly representable in fp32 (test setup)"
    bad = got.double() != want
    if bool(bad.any()):
        idx = bad.nonzero()[0].tolist()
        d = (got.double() - want).abs().nan_to_num(float("inf")).max().item()
        pytest.fail(f"{what}: {int(bad.sum())} of {got.numel()} elements differ from the fp64 reference, max |d| {d:.6g}, "
                    f"first at {idx}: got {got[tuple(idx)].item()!r}, want {want[tuple(idx)].item()!r}")


def _expect_tc(mode, kind, K, cout):
    """whether the forward call takes conv_plan_tc (capi.cu tc_ok; a deconvolution needs one parent per fine site)"""
    return mode != "fp32" and cout % 32 == 0 and cout <= 256 and not (kind == "deconv" and K == 64)


def _inputs(case, seed=0):
    kind, level, K, cin, cout = case
    rs = np.random.RandomState(seed + 7 * cin + 13 * cout + K + sum(map(ord, kind + level)))
    lv = _level(level)
    g = _geom(lv, kind, K)
    x = grid_x(rs, g["n_src"], cin)
    w = grid_w(rs, cin, cout) if kind == "nin" else grid_w(rs, K, cin, cout)
    dy = grid_w(rs, g["n_dst"], cout)
    return lv, g, x, w, dy


# ------------------------------------------------------------------ 1. forward, input gradient and weight gradient, bitwise
FWD_CASES = [
    # submanifold 3^3 on the small building (40 tiles: the filter offsets are split over CTAs)
    ("subm", "small", 27, 9, 32), ("subm", "small", 27, 16, 64), ("subm", "small", 27, 20, 64), ("subm", "small", 27, 32, 32),
    ("subm", "small", 27, 48, 256), ("subm", "small", 27, 64, 48), ("subm", "small", 27, 96, 96), ("subm", "small", 27, 128, 160),
    ("subm", "small", 27, 192, 192), ("subm", "small", 27, 256, 256), ("subm", "small", 27, 64, 16), ("subm", "small", 1, 32, 128),
    ("subm", "small", 1, 256, 128),
    # a mid-size level (111 tiles, one CTA per item) and level 0 of the 300 x 280 x 40 building (many super-tiles)
    ("subm", "mini4", 27, 64, 64), ("subm", "big", 27, 16, 64), ("subm", "big", 27, 32, 32), ("subm", "big", 27, 128, 128),
    ("subm", "big", 27, 96, 256),
    # strided convolution (K = 8, K = 64), z-collapse (K = 16), deconvolution (per-tile weight slice)
    ("conv", "small", 8, 32, 64), ("conv", "small", 8, 128, 128), ("conv", "small", 64, 32, 64), ("conv", "small", 64, 64, 256),
    ("conv", "small", 16, 32, 64), ("conv", "big", 8, 64, 128),
    ("deconv", "small", 8, 32, 64), ("deconv", "small", 8, 128, 128), ("deconv", "small", 8, 20, 32), ("deconv", "small", 64, 64, 32),
    ("deconv", "big", 8, 128, 64),
    # NetworkInNetwork (dense rows, no plan)
    ("nin", "small", 1, 64, 128), ("nin", "rows1", 1, 9, 32), ("nin", "rows129", 1, 192, 96),
    # ragged single tiles
    ("subm", "rows1", 27, 64, 64), ("subm", "rows77", 27, 32, 64), ("subm", "rows128", 27, 64, 128), ("subm", "rows129", 27, 128, 64),
]


def _cid(c):
    return "-".join(map(str, c))


@pytest.mark.parametrize("case", FWD_CASES, ids=_cid)
@pytest.mark.parametrize("mode", list(MODES))
def test_exact_grid_bitwise(mode, case):
    """Forward, input gradient and weight gradient of one layer in one math mode equal the fp64 reference bit for bit.  Layers whose
    input rows are not a multiple of 64 channels run after a 256-channel layer on the same stream, so the scratch buffers that hold
    their padded operand copies start out full of non-zero data."""
    if mode != "fp32":
        _tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, dy = _inputs(case)
    want = ref_forward(lv, kind, g, x, w)
    try:
        _set_mode(mode)
        if cin % 64 and kind != "nin" and mode != "fp32":
            rs = np.random.RandomState(1)
            gs = _geom(lv, "subm", 27)
            run_forward(lv, "subm", gs, torch.from_numpy(rs.randn(lv.n, 256).astype(np.float32)).cuda(), grid_w(rs, 27, 256, 256))
        before = _counters()
        out, _ = run_forward(lv, kind, g, x, w)
        d = _delta(before)
        print(f"[exact] {mode} {_cid(case)} forward: {d}")
        assert_exact(out, want, f"{mode} {_cid(case)} forward")
        tc = _expect_tc(mode, kind, K, cout)
        assert d["tc"] == int(tc) and d["simt"] == int(not tc), d
        assert d["x3"] == int(tc and mode == "tf32x3"), d
        if kind == "nin":
            return
        before = _counters()
        d_in, dw = run_backward(lv, kind, g, x, dy, w)
        d = _delta(before)
        print(f"[exact] {mode} {_cid(case)} backward: {d}")
        want_din, want_dw = ref_backward(lv, kind, g, x, dy, w)
        assert_exact(d_in, want_din, f"{mode} {_cid(case)} input gradient")
        assert_exact(dw, want_dw, f"{mode} {_cid(case)} weight gradient")
    finally:
        _set_mode("fp32")


# ------------------------------------------------------------------ 2. fused epilogue: bias, add, bf16 copy, lateral stage, statistics
EPI_CASES = [  # (case, bias, addend)
    (("subm", "small", 27, 64, 64), True, True), (("subm", "mini4", 27, 128, 128), True, True), (("subm", "big", 27, 32, 32), False, True),
    (("conv", "small", 8, 64, 128), True, False), (("deconv", "small", 8, 128, 64), False, True), (("nin", "mini4", 1, 32, 64), True, False),
]


@pytest.mark.parametrize("case,bias,addend", EPI_CASES, ids=lambda v: _cid(v) if isinstance(v, tuple) else str(v))
@pytest.mark.parametrize("mode", TC_MODES)
def test_fused_epilogue_exact(mode, case, bias, addend):
    """bias and the fused add (out = conv + addend) in the epilogue, and the bf16 output copy, which must equal out.to(bfloat16)"""
    _tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, _ = _inputs(case, seed=1)
    rs = np.random.RandomState(cin + cout)
    b = grid_w(rs, cout) if bias else None
    ad = grid_w(rs, g["n_dst"], cout) if addend else None
    want = ref_forward(lv, kind, g, x, w, b, ad)
    try:
        _set_mode(mode)
        before = _counters()
        out, o16 = run_forward(lv, kind, g, x, w, b, ad, want16=kind != "nin")
        d = _delta(before)
    finally:
        _set_mode("fp32")
    print(f"[epilogue] {mode} {_cid(case)} bias={bias} add={addend}: {d}")
    assert d["tc"] == 1 and d["simt"] == 0, d
    assert_exact(out, want, f"{mode} {_cid(case)} epilogue")
    if o16 is not None:
        assert torch.equal(o16.view(torch.int16), out.to(torch.bfloat16).view(torch.int16)), "bf16 copy differs from out.to(bfloat16)"


def _stats_sums(stats, c):
    s = stats.view(8, 2, 128).sum(0)
    return s[0, :c], s[1, :c]


@pytest.mark.parametrize("c_lat", [32, 64, 128])
@pytest.mark.parametrize("kind,level", [("subm", "mini4"), ("deconv", "small"), ("subm", "big")])
@pytest.mark.parametrize("mode", TC_MODES)
def test_lateral_stage_and_epilogue_stats_exact(mode, kind, level, c_lat):
    """out = conv(x) + y[row] @ W_lat in one launch (the lateral stage, pseudo filter offset 63), with the per-channel sum and sum
    of squares of out accumulated by the epilogue.  The statistics are fp32 per lane before the double atomics: with sparse inputs
    every partial sum stays a multiple of 1/64 below 2^18, so they equal the fp64 sums bitwise too (asserted as a precondition)."""
    _tc_or_skip()
    lv = _level(level)
    K = 27 if kind == "subm" else 8
    g = _geom(lv, kind, K)
    C0, n = 64, g["n_dst"]
    rs = np.random.RandomState(c_lat + K)
    density = 0.01 if level == "big" else 0.1
    x, w = grid_x(rs, g["n_src"], C0, density), grid_w(rs, K, C0, C0)
    y, wl = grid_x(rs, n, c_lat, density), grid_w(rs, c_lat, C0)
    want = ref_forward(lv, kind, g, x, w) + y.double() @ wl.double()
    s1, s2 = want.sum(0), (want * want).sum(0)
    lib = _lib()
    try:
        _set_mode(mode)
        stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
        y16 = y.to(torch.bfloat16)
        before = _counters()
        _check(lib.scn_fuse_next_lateral(_p(y), _p(y16), _p(wl), 0, c_lat, n))
        _check(lib.scn_fuse_next_stats(_p(stats)))
        out, _ = run_forward(lv, kind, g, x, w)
        took_l, took_s = C.c_int(), C.c_int()
        _check(lib.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
        d = _delta(before)
    finally:
        _set_mode("fp32")
    print(f"[lateral] {mode} {kind} {level} c_lat={c_lat}: {d}, stats taken {took_s.value}")
    assert took_l.value == 1 and d["lateral"] == 1, d
    assert_exact(out, want, f"{mode} {kind} {level} lateral {c_lat}")
    if d["split"] == 0:
        assert took_s.value == 1 and d["stats"] == 1, d
        assert float(want.abs().sum(0).max()) < 2 ** 21 and float(s2.max()) < 2 ** 18, "statistics would not be exact in fp32 (test setup)"
        got1, got2 = _stats_sums(stats, C0)
        assert_exact(got1, s1, "epilogue sum")
        assert_exact(got2, s2, "epilogue sum of squares")
    else:
        assert took_s.value == 0


# ------------------------------------------------------------------ 3. weight gradient: which kernel, every shape branch
def _dw_tc_ok(cin, cout, K):  # restates dw_tc_ok (conv_tc.cu) for the bf16 mode
    return not ((cin % 32 and cin > 32) or cin > 256 or (cin > 128 and cin % 128) or cout % 32 or cout > 256 or ((cin + 127) // 128) * cout > 512 or K > 64)


DW_CASES = [
    ("subm", "small", 27, 9, 32), ("subm", "small", 27, 20, 64), ("subm", "small", 27, 32, 128), ("subm", "mini4", 27, 64, 256),
    ("subm", "small", 27, 128, 128), ("subm", "small", 27, 256, 256), ("subm", "small", 27, 256, 32), ("subm", "big", 27, 32, 32),
    ("conv", "small", 8, 32, 64), ("conv", "small", 64, 64, 32), ("conv", "small", 16, 128, 64), ("deconv", "small", 8, 64, 128),
    ("deconv", "small", 8, 9, 32), ("subm", "lines", 27, 32, 32), ("subm", "lines", 27, 256, 64),
    ("subm", "small", 27, 48, 64), ("subm", "small", 27, 64, 16),   # rejected by dw_tc_ok: the CUDA-core k_dw
]


@pytest.mark.parametrize("case", DW_CASES, ids=_cid)
def test_weight_gradient_kernel_and_exactness(case):
    """bf16 mode: d_W on conv_dw_tc (R = 128 / 64 rules per stage, nMh = 2 for 256 input channels, one or two accumulators, 32- and
    64-byte rows, lists short enough that parts of them are empty) or, for the shapes dw_tc_ok rejects, on the CUDA-core k_dw.  Which
    one ran is read from the float-atomic counter: conv_dw_tc is one launch per call, k_dw one per non-empty rule list."""
    _tc_or_skip()
    kind, level, K, cin, cout = case
    lv, g, x, w, dy = _inputs(case, seed=2)
    _, want_dw = ref_backward(lv, kind, g, x, dy, w)
    nonempty = sum(int(len(r) > 0) for r in lv.rules(g["key"]))
    try:
        _set_mode("bf16")
        before = _counters()
        _, dw = run_backward(lv, kind, g, x, dy, w, want_din=kind != "subm")
        d = _delta(before)
    finally:
        _set_mode("fp32")
    tc = _dw_tc_ok(cin, cout, K)
    launches = d["atomic"] - d["split"]  # (a split input-gradient launch also accumulates atomically)
    print(f"[dw] {_cid(case)}: {'conv_dw_tc' if launches == 1 else 'k_dw'} ({launches} float-atomic launches, {nonempty} non-empty lists), {d}")
    assert launches == (1 if tc else nonempty), (launches, nonempty, d)
    if tc and cin % 32 == 0:
        assert d["reused"] >= 1, d  # the bf16 copy of d_out made for the input gradient is reused
    assert_exact(dw, want_dw, f"bf16 {_cid(case)} weight gradient")


# ------------------------------------------------------------------ 4. deterministic mode
@pytest.fixture
def det():
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn)


@pytest.mark.parametrize("mode", TC_MODES)
def test_deterministic_mode_exact(mode):
    """The split-offset partials (k_split_sum), the tiles of a large level and the bf16 weight gradient's ordered parts: with
    torch.use_deterministic_algorithms(True) the results equal the default mode's and the reference bit for bit."""
    _tc_or_skip()
    cases = [("subm", "small", 27, 64, 64), ("subm", "big", 27, 32, 32), ("deconv", "small", 8, 128, 64)]
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        _set_mode(mode)
        for case in cases:
            kind = case[0]
            lv, g, x, w, dy = _inputs(case, seed=3)
            want = ref_forward(lv, kind, g, x, w)
            want_din, want_dw = ref_backward(lv, kind, g, x, dy, w)
            res = []
            for flag in (False, True):
                torch.use_deterministic_algorithms(flag)
                out, o16 = run_forward(lv, kind, g, x, w, want16=True)
                res.append((out, o16) + run_backward(lv, kind, g, x, dy, w))
            torch.use_deterministic_algorithms(on, warn_only=warn)
            for (out, o16, d_in, dw), tag in zip(res, ("default", "deterministic")):
                assert_exact(out, want, f"{mode} {tag} {_cid(case)} forward")
                assert torch.equal(o16.view(torch.int16), out.to(torch.bfloat16).view(torch.int16))
                assert_exact(d_in, want_din, f"{mode} {tag} {_cid(case)} input gradient")
                assert_exact(dw, want_dw, f"{mode} {tag} {_cid(case)} weight gradient")
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn)
        _set_mode("fp32")


# ------------------------------------------------------------------ 5. every launcher knob, one subprocess each
VARIANT_FWD = [("subm", "small", 27, 64, 64), ("subm", "mini4", 27, 64, 64), ("subm", "big", 27, 32, 32), ("subm", "big", 27, 64, 64),
               ("conv", "small", 64, 32, 64), ("deconv", "small", 8, 128, 128), ("subm", "small", 27, 256, 256)]
VARIANT_DW = [("subm", "small", 27, 64, 64), ("subm", "lines", 27, 32, 32)]
KNOBS = [
    {"SCN_TC_CTAS": "1", "SCN_DW_PLAN": "1", "SCN_DW_ITEMS": "1"},
    {"SCN_TC_CTAS": "2", "SCN_DW_PLAN": "1", "SCN_DW_ITEMS": "48"},
    {"SCN_TC_T": "1", "SCN_DW_PART": "64"},
    {"SCN_TC_T": "2"}, {"SCN_TC_T": "3"}, {"SCN_TC_T": "4"},
    {"SCN_TC_S": "2", "SCN_TC_LAG": "0"},
    {"SCN_TC_PW8": "1"}, {"SCN_TC_PW8": "2"}, {"SCN_TC_PW8": "3"},
    {"SCN_TC_SPLIT_MAX": "0"}, {"SCN_TC_SPLIT_MAX": "100000", "SCN_TC_SMALL_ONE": "0"},  # (two CTAs per SM: the 111 tiles of mini4 then split)
]


def _variant_name(mode, case):
    return f"{mode}-{_cid(case)}"


def variant_child(out_dir):
    """Body of the knob subprocesses: the VARIANT_* cases on the exact grid, results saved as .npy; a [case] line on stderr names
    the case whose [tcprof] lines follow, a [cnt] line gives its counter deltas."""
    def mark(name, d):
        print(f"[cnt] {name} " + " ".join(f"{k}={v}" for k, v in d.items()), file=sys.stderr, flush=True)
    for case in VARIANT_FWD:
        for mode in TC_MODES:
            name = _variant_name(mode, case)
            print(f"[case] {name}", file=sys.stderr, flush=True)
            lv, g, x, w, _ = _inputs(case, seed=4)
            _set_mode(mode)
            before = _counters()
            out, _ = run_forward(lv, case[0], g, x, w)
            mark(name, _delta(before))
            np.save(os.path.join(out_dir, name + ".npy"), out.cpu().numpy())
    for case in VARIANT_DW:
        name = _variant_name("dw", case)
        print(f"[case] {name}", file=sys.stderr, flush=True)
        lv, g, x, w, dy = _inputs(case, seed=4)
        _set_mode("bf16")
        before = _counters()
        _, dw = run_backward(lv, case[0], g, x, dy, w, want_din=False)
        mark(name, _delta(before))
        np.save(os.path.join(out_dir, name + ".npy"), dw.cpu().numpy())
    _set_mode("fp32")


_CHILD = r"""
import os, sys
sys.path[:0] = [{root!r}, os.path.join({root!r}, "tests")]
import test_gpu_tc_exact as t
t.variant_child({out!r})
"""

_REFS = {}


def _variant_ref(name, case):
    if name not in _REFS:
        lv, g, x, w, dy = _inputs(case, seed=4)
        _REFS[name] = ref_backward(lv, case[0], g, x, dy, w)[1] if name.startswith("dw-") else ref_forward(lv, case[0], g, x, w)
    return _REFS[name]


def _parse_child(stderr):
    """{case name: ([tcprof] dicts, counter dict)}"""
    res, cur = {}, None
    for line in stderr.splitlines():
        if line.startswith("[case] "):
            cur = line.split()[1]
            res[cur] = ([], {})
        elif line.startswith("[tcprof]") and cur:
            res[cur][0].append({k: int(v) for k, v in re.findall(r"(\w+)=(-?\d+)", line.split("|")[0])})
        elif line.startswith("[cnt] ") and cur:
            res[cur][1].update({k: int(v) for k, v in re.findall(r"(\w+)=(-?\d+)", line)})
    return res


@pytest.mark.parametrize("knobs", KNOBS, ids=lambda k: ",".join(f"{a}={b}" for a, b in k.items()))
def test_launcher_variant(tmp_path, knobs):
    """One process per knob setting (each knob is read once per process).  SCN_TC_PROF=1 makes the launcher print its configuration
    per launch ([tcprof] ctas, pw, T, S, lag, nAcc, kSplit): the setting must show there, or in the plan-driven weight-gradient
    counter (13) and the split counter (9); and every result equals the fp64 reference bit for bit."""
    _tc_or_skip()
    env = dict(os.environ, SCN_TC_PROF="1", **knobs)
    r = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, out=str(tmp_path))], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    seen = _parse_child(r.stderr)
    cases = {_variant_name(m, c): c for c in VARIANT_FWD for m in TC_MODES}
    cases.update({_variant_name("dw", c): c for c in VARIANT_DW})
    names = list(cases)
    assert sorted(seen) == sorted(names), sorted(seen)
    for name, case in cases.items():
        assert_exact(torch.from_numpy(np.load(tmp_path / (name + ".npy"))).cuda(), _variant_ref(name, case), f"{knobs} {name}")
    prof = {n: v[0] for n, v in seen.items()}
    cnt = {n: v[1] for n, v in seen.items()}
    fwd = [n for n in names if not n.startswith("dw-")]
    lines = [(n, p) for n in fwd for p in prof[n]]
    assert all(len(prof[n]) == 1 for n in fwd), {n: len(prof[n]) for n in fwd}
    for n, p in lines:
        print(f"[variant] {knobs} {n}: " + " ".join(f"{k}={v}" for k, v in p.items() if k in ("ctas", "pw", "T", "S", "lag", "nAcc", "kSplit")))
    x3 = lambda n: n.startswith("tf32x3")
    two_cta = lambda n, p: not x3(n) and p["Cout"] <= 128
    if knobs.get("SCN_TC_CTAS") == "1":
        assert all(p["ctas"] == 1 for n, p in lines if not (n.startswith("bf16") and p["Cin"] == 32)), lines  # (packed rows: two CTAs)
    if knobs.get("SCN_TC_CTAS") == "2":
        assert all(p["ctas"] == 2 for n, p in lines if two_cta(n, p)) and any(p["ctas"] == 2 and "small" in n for n, p in lines), lines
    if "SCN_TC_T" in knobs:
        t = int(knobs["SCN_TC_T"])
        tiled = [(n, p) for n, p in lines if "deconv" not in n]  # (deconvolution plans: one tile per item)
        assert all(p["T"] <= t for n, p in tiled) and any(p["T"] == t for n, p in tiled), tiled
    if "SCN_TC_S" in knobs:
        assert all(p["S"] == 2 for n, p in lines), lines
    if "SCN_TC_LAG" in knobs:
        assert all(p["lag"] == 0 for n, p in lines), lines
    if "SCN_TC_PW8" in knobs:
        bits = int(knobs["SCN_TC_PW8"])
        for n, p in lines:
            if p["ctas"] == 2:
                packed = n.startswith("bf16") and p["Cin"] == 32
                assert p["pw"] == (8 if bits & (1 if packed else 2) else 4), (n, p)
        assert any(p["ctas"] == 2 and p["pw"] == 8 for n, p in lines), lines
    if knobs.get("SCN_TC_SMALL_ONE") == "0":
        assert all(p["ctas"] == 2 for n, p in lines if "small" in n and two_cta(n, p)), lines
    if knobs.get("SCN_TC_SPLIT_MAX") == "0":
        assert all(p["kSplit"] == 1 for n, p in lines) and all(cnt[n]["split"] == 0 for n in fwd), lines
    if knobs.get("SCN_TC_SPLIT_MAX") == "100000":
        assert all(p["kSplit"] > 1 for n, p in lines if "mini4" in n and not x3(n)), lines
    elif "SCN_TC_T" not in knobs:  # (a forced T changes the number of items)
        assert all(p["kSplit"] == 1 for n, p in lines if "mini4" in n), lines
    dw = [n for n in names if n.startswith("dw-")]
    assert all(cnt[n]["dw_plan"] == int(knobs.get("SCN_DW_PLAN") == "1") for n in dw), {n: cnt[n] for n in dw}


# ------------------------------------------------------------------ 6. operand rounding conventions (single products)
def _tf32(x, how):
    b = x.contiguous().view(torch.int32)
    if how == "trunc":
        r = b & -8192
    elif how == "rna":
        r = (b + 0x1000) & -8192
    else:  # rne
        r = (b + 0xFFF + ((b >> 13) & 1)) & -8192
    return r.view(torch.float32)


def _bf16(x, how):
    b = x.contiguous().view(torch.int32)
    if how == "trunc":
        r = b & -65536
    elif how == "rna":
        r = (b + 0x8000) & -65536
    else:
        return x.to(torch.bfloat16).float()
    return r.view(torch.float32)


def _probe_values(rs, n, low_bits):
    """fp32 values with random mantissas; a quarter are exact ties of rounding away `low_bits` bits, a quarter one ulp off a tie"""
    m = rs.randint(0, 1 << 23, n).astype(np.int64)
    half = 1 << (low_bits - 1)
    q = n // 4
    m[:q] = (m[:q] & ~((1 << low_bits) - 1)) | half
    m[q:2 * q] = (m[q:2 * q] & ~((1 << low_bits) - 1)) | (half + rs.choice([-1, 1], q))
    bits = (rs.randint(124, 131, n).astype(np.int64) << 23) | m | (rs.randint(0, 2, n).astype(np.int64) << 31)
    return torch.from_numpy(bits.astype(np.uint32).view(np.float32).copy()).cuda()


@pytest.mark.parametrize("mode,cin", [("tf32", 32), ("tf32", 9), ("tf32", 20), ("bf16", 64), ("bf16", 9), ("bf16", 20)])
def test_operand_rounding_convention(mode, cin):
    """One active channel per row (a NetworkInNetwork of 128 rows, 32 outputs), so every output is ONE product of two rounded
    operands, exact in fp32.  With the other operand exact, each output shows how one operand was rounded, ties included:
    tf32 weights cvt.rna; tf32 activation rows as the tensor core reads them (TF32_ACT); bf16 activations and weights round to
    nearest even, through k_to_bf16 (64 channels) and through the zero-padding copy k_pad_rows_bf16 (9 and 20 channels)."""
    _tc_or_skip()
    n, cout = 128, 32
    rs = np.random.RandomState(cin)
    low = 13 if mode == "tf32" else 16
    rnd = _tf32 if mode == "tf32" else _bf16
    ch = torch.from_numpy(np.arange(n) % cin).cuda()
    lv = _level("rows1")  # (dense rows: no Metadata involved)
    g = dict(n_src=n, n_dst=n)
    found = {}
    for operand in ("act", "weight"):
        a = _probe_values(rs, n, low) if operand == "act" else torch.from_numpy(rs.choice([-2.0, -1.0, 1.0, 2.0], n).astype(np.float32)).cuda()
        w = (_probe_values(rs, cin * cout, low) if operand == "weight" else rnd(_probe_values(rs, cin * cout, low), "rne")).view(cin, cout)
        x = torch.zeros(n, cin, device="cuda")
        x[torch.arange(n, device="cuda"), ch] = a
        try:
            _set_mode(mode)
            before = _counters()
            out, _ = run_forward(lv, "nin", g, x, w)
            assert _delta(before)["tc"] == 1
        finally:
            _set_mode("fp32")
        match = []
        for how in ("trunc", "rna", "rne"):
            ra, rw = (rnd(a, how), w) if operand == "act" else (a, rnd(w, how))
            if torch.equal(out.double(), ra.double()[:, None] * rw.double()[ch]):
                match.append(how)
        found[operand] = match
    print(f"[rounding] {mode} Cin={cin}: activations {found['act']}, weights {found['weight']}")
    want_act = TF32_ACT if mode == "tf32" else "rne"
    want_w = "rna" if mode == "tf32" else "rne"
    assert found["act"] == [want_act] and found["weight"] == [want_w], found


# ------------------------------------------------------------------ 7. accumulation error on random data
BOUND_CASES = [("subm", "small", 27, 64, 64), ("subm", "big", 27, 128, 128), ("subm", "small", 27, 256, 256), ("conv", "small", 8, 96, 128),
               ("nin", "mini4", 1, 192, 64)]


def _rounded_terms(mode, cin, x, w):
    """[(A, W)] whose fp64 products summed give ref_r: the operands exactly as the kernel rounds them"""
    if mode == "fp32":
        return [(x, w)]
    if mode == "tf32x3":  # hi = tf32(v), lo = tf32(v - hi); the kernel drops lo * lo
        xh, wh = _tf32(x, "rna"), _tf32(w, "rna")
        xl, wl = _tf32(x - xh, "rna"), _tf32(w - wh, "rna")
        return [(xh, wh), (xh, wl), (xl, wh)]
    if mode == "bf16" and (cin % 64 == 0 or cin in (16, 32) or cin < 32):
        return [(_bf16(x, "rne"), _bf16(w, "rne"))]
    return [(_tf32(x, TF32_ACT), _tf32(w, "rna"))]  # tf32 mode, and bf16 mode with TF32 operands (e.g. 96 channels)


@pytest.mark.parametrize("mode", list(MODES))
def test_accumulation_error_bound(mode):
    """N(0, 1) data: max over outputs of |got - ref_r| / S <= TAU[mode], with ref_r the fp64 sum of the rounded operands' products
    and S the fp64 sum of their magnitudes, so what is left is the fp32 accumulation inside the kernel.  For tf32x3 the bound also
    holds against ref_r without the dropped lo * lo term: that term and the accumulation are the whole of its error floor."""
    if mode != "fp32":
        _tc_or_skip()
    worst = 0.0
    for case in BOUND_CASES:
        kind, level, K, cin, cout = case
        lv = _level(level)
        g = _geom(lv, kind, K)
        rs = np.random.RandomState(cin + cout)
        x = torch.from_numpy(rs.randn(g["n_src"], cin).astype(np.float32)).cuda()
        w = torch.from_numpy((rs.randn(*((cin, cout) if kind == "nin" else (K, cin, cout))) * (1 / (cin * K)) ** 0.5).astype(np.float32)).cuda()
        try:
            _set_mode(mode)
            out, _ = run_forward(lv, kind, g, x, w)
        finally:
            _set_mode("fp32")
        terms = _rounded_terms(mode, cin, x, w)
        ref_r = sum(ref_forward(lv, kind, g, a, b) for a, b in terms)
        S = sum(ref_forward(lv, kind, g, a.abs(), b.abs()) for a, b in terms)
        ratio = float(((out.double() - ref_r).abs() / S.clamp_min(1e-300)).max())
        exact = float((ref_forward(lv, kind, g, x, w) - ref_r).abs().max() / ref_r.abs().max())
        print(f"[bound] {mode} {_cid(case)}: max |got - ref_r| / S = {ratio:.3e} ({ratio * 2 ** 24:.2f} x 2^-24); "
              f"operand rounding alone {exact:.2e} of max|out|")
        worst = max(worst, ratio)
    print(f"[bound] {mode}: worst {worst:.3e}, tau {TAU[mode]:.3e}")
    assert worst <= TAU[mode], (worst, TAU[mode])
    if mode == "tf32x3":  # the split adds no error of its own: what is left fits the bound of plain tf32 accumulation
        assert worst <= TAU["tf32"], (worst, TAU["tf32"])
