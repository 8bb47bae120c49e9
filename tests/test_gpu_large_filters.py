"""Filters of more than 64 offsets (5^3, 7^3, 8^3, [1, 1, z] up to z = 512): rulebooks, the chunked tensor-core launches and the
CUDA-core paths that serve them (DESIGN.md sections 4.3, 4.4 and 7).

A plan of K > 64 offsets is stored chunk-major and runs as ceil(K / 63) launches of the unchanged conv_plan_tc, one per chunk of
<= 63 offsets; scn_debug_counter(16) counts those launches, so every tensor-core case below proves the chunked path ran and the
CUDA-core fallback did not.

CPU part: the oracle (oracle/scn_oracle.c) against the reference's compiled Metadata (skipped where oracle/_ref is absent).
GPU part: rulebooks bit-exact against the oracle; forward, input gradient and weight gradient bit for bit against the fp64
gather-GEMM on the exact grid of test_gpu_tc_exact.py in all four math modes; the fused epilogue; per-layer tolerances on N(0, 1)
data; deterministic mode; FPN_Net end to end with 5^3 / 2 downsampling and a [1, 1, 128] z-collapse."""
import numpy as np
import pytest
import torch

import fpn_util
import test_gpu_tc_exact as tx
from detection_3d_b200 import synthetic
from oracle import scn_oracle as so

CNT = dict(tx.CNT, chunk=16, lateral_fallback=6, train_replay=11)
SHAPES = {  # filter, stride; "zc" = [1, 1, z] over the whole z extent of the level (z-collapse), stride 1
    "5": ([5, 5, 5], [1, 1, 1]), "7": ([7, 7, 7], [1, 1, 1]), "8": ([8, 8, 8], [1, 1, 1]), "z128": ([1, 1, 128], [1, 1, 1]),
    "5s2": ([5, 5, 5], [2, 2, 2]), "7s2": ([7, 7, 7], [2, 2, 2]), "5s5": ([5, 5, 5], [5, 5, 5]),
}
# per layer, rtol and atol x max|ref| (DESIGN.md section 7)
LAYER_TOL = {"fp32": (2e-4, 2e-5), "tf32x3": (2e-4, 2e-5), "tf32": (4e-3, 2e-3), "bf16": (1.6e-2, 8e-3)}


def _chunks(K):
    return 1 if K <= 64 else (K + 62) // 63


def _level_coords(name):
    """(coords [n, 4], spatial size) of a level: the small building, a z-collapse grid of depth z, two batch items, one site"""
    small = synthetic.small_building(40, 36, 12, 3, seed=4)
    if name == "small":
        return small, [64, 64, 32]
    if name.startswith("zc"):
        return small, [64, 64, int(name[2:])]
    if name == "batch2":
        b = synthetic.small_building(30, 28, 10, 2, seed=8)
        b[:, 3] = 1
        return np.concatenate([small, b]), [64, 64, 32]
    if name == "mini4":  # above kSortMinSites: the submanifold plan is sorted by neighbour class
        return synthetic.building_coords(nx=60, ny=56, nz=24, n_walls=3, seed=3), [64, 64, 32]
    assert name == "rows1"
    return np.array([[3, 4, 5, 0]], np.int64), [16, 16, 16]


class _WLevel(tx._Level):
    def __init__(self, name):
        from gpu_adapter import GpuMetadata
        self.coords, self.full = _level_coords(name)
        self.G = GpuMetadata()
        self.n = self.G.input_layer(self.full, self.coords, 0, 4)
        self._O, self._rules, self._made, self._o_made = None, {}, [], set()


_WLEVELS = {}


def _wlevel(name):
    if name not in _WLEVELS:
        _WLEVELS[name] = _WLevel(name)
    return _WLEVELS[name]


def _wgeom(lv, kind, shape):
    """as tx._geom: `a` is the finer grid; the layer reads rows of `src` and writes rows of `dst`"""
    full = lv.full
    if kind == "subm":
        f = SHAPES[shape][0]
        return dict(a=full, b=full, f=f, s=[1, 1, 1], n_src=lv.n, n_dst=lv.n, key=("subm", tuple(f)), K=int(np.prod(f)))
    if shape == "zc":
        a, b, f, s = full, [full[0], full[1], 1], [1, 1, full[2]], [1, 1, 1]
    else:
        f, s = SHAPES[shape]
        a, b = full, [(full[d] - f[d]) // s[d] + 1 for d in range(3)]
    lv.make_conv(a, b, f, s)
    na, nb = lv.nactive(a), lv.nactive(b)
    g = dict(a=a, b=b, f=f, s=s, key=("conv", tuple(a), tuple(b), tuple(f), tuple(s)), K=int(np.prod(f)))
    return dict(g, n_src=na, n_dst=nb) if kind == "conv" else dict(g, n_src=nb, n_dst=na)


def _counters():
    return {k: tx._lib().scn_debug_counter(i) for k, i in CNT.items()}


def _delta(before):
    now = _counters()
    return {k: now[k] - before[k] for k in now}


def _forward_on_tc(mode, kind, g, cout, n_src_rows):
    """(tensor-core launches, chunked launches) a forward must show: capi.cu tc_ok, one parent per fine site for a deconvolution"""
    if mode == "fp32" or cout % 32 or n_src_rows == 0:
        return 0, 0
    if kind == "deconv":
        single = g["f"] == g["s"] or (g["f"][0] == 1 and g["f"][1] == 1 and g["s"] == [1, 1, 1])
        return (1, 0) if single else (0, 0)
    return _chunks(g["K"]), _chunks(g["K"]) if g["K"] > 64 else 0


# ------------------------------------------------------------------ CPU: the oracle against the reference's own Metadata
@pytest.mark.skipif(not so.have_ref(), reason="reference build only exists in the build container")
@pytest.mark.parametrize("batch", [1, 2])
def test_oracle_wide_rulebooks_match_reference(batch):
    rs = np.random.RandomState(batch)
    n = 3000
    c = np.stack([rs.randint(0, 40, n), rs.randint(0, 40, n), rs.randint(0, 20, n)], 1).astype(np.int64)
    c = np.concatenate([c, np.sort(rs.randint(0, batch, (n, 1)), 0)], 1)
    full = [64, 64, 32]
    for sub in ([5, 5, 5], [7, 7, 7], [1, 1, 128]):
        O, R = so.OracleMetadata(), so.RefMetadata()
        assert O.input_layer(full, c, batch, 4) == R.input_layer(full, c, batch, 4)
        for a, b in zip(O.submanifold_rules(full, sub), R.submanifold_rules(full, sub)):
            assert np.array_equal(a, b), sub
    for z in (96, 128, 512):
        fz = [64, 64, z]
        O, R = so.OracleMetadata(), so.RefMetadata()
        O.input_layer(fz, c, batch, 4), R.input_layer(fz, c, batch, 4)
        for a, b in zip(O.conv_rules(fz, [64, 64, 1], [1, 1, z], [1, 1, 1]), R.conv_rules(fz, [64, 64, 1], [1, 1, z], [1, 1, 1])):
            assert np.array_equal(a, b), z
    for f in (5, 7):
        O, R = so.OracleMetadata(), so.RefMetadata()
        O.input_layer(full, c, batch, 4), R.input_layer(full, c, batch, 4)
        out = [(v - f) // 2 + 1 for v in full]
        for a, b in zip(O.conv_rules(full, out, [f] * 3, [2] * 3), R.conv_rules(full, out, [f] * 3, [2] * 3)):
            assert np.array_equal(a, b), f
        assert np.array_equal(O.spatial_locations(out), R.spatial_locations(out))


# ------------------------------------------------------------------ GPU: rulebooks bit-exact against the oracle
RB_CASES = [("subm", lvl, sh) for lvl in ("rows1", "small", "mini4", "batch2") for sh in ("5", "7", "z128")] + \
           [("subm", "small", "8")] + \
           [("conv", lvl, sh) for lvl in ("rows1", "small", "mini4", "batch2") for sh in ("5s2", "7s2")] + \
           [("conv", f"zc{z}", "zc") for z in (96, 128, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,level,shape", RB_CASES, ids=lambda v: str(v))
def test_gpu_rulebooks_bit_exact(kind, level, shape):
    """Every list of the GPU rulebook equals the oracle's, in the reference's order: plan, first-touch numbering and list
    positions of filters beyond 64 offsets.  Fresh Metadata per case, so the lists are built on demand from the plan."""
    from gpu_adapter import GpuMetadata
    coords, full = _level_coords(level)
    G, O = GpuMetadata(), so.OracleMetadata()
    assert G.input_layer(full, coords, 0, 4) == O.input_layer(full, coords, 0, 4)
    if kind == "subm":
        f = SHAPES[shape][0]
        got, want = G.submanifold_rules(full, f), O.submanifold_rules(full, f)
    else:
        if shape == "zc":
            out, f, s = [full[0], full[1], 1], [1, 1, full[2]], [1, 1, 1]
        else:
            f, s = SHAPES[shape]
            out = [(full[d] - f[d]) // s[d] + 1 for d in range(3)]
        got, want = G.conv_rules(full, out, f, s), O.conv_rules(full, out, f, s)
        assert np.array_equal(G.spatial_locations(out), O.spatial_locations(out)), "output numbering"
    assert len(got) == len(want) == int(np.prod(f))
    for k, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a.reshape(-1), np.asarray(b).reshape(-1)), (kind, level, shape, k)


@pytest.mark.gpu
def test_limits_raise_naming_them():
    """A filter volume above 512, and more than 64 output cells per input site (5^3 with stride 1), keep raising."""
    from gpu_adapter import GpuMetadata
    coords, full = _level_coords("small")
    G = GpuMetadata()
    G.input_layer(full, coords, 0, 4)
    with pytest.raises(Exception, match="512"):
        G.submanifold_rules(full, [9, 9, 9])
    with pytest.raises(Exception, match="64"):
        G.conv_rules(full, [60, 60, 28], [5, 5, 5], [1, 1, 1])


# ------------------------------------------------------------------ GPU: exact grid, bit for bit
EXACT_CASES = [
    ("subm", "small", "5", 32, 64), ("subm", "small", "7", 64, 32), ("subm", "small", "z128", 32, 32), ("subm", "mini4", "5", 64, 64),
    ("subm", "rows1", "5", 32, 32), ("subm", "batch2", "5", 16, 64),
    ("conv", "small", "5s2", 32, 64), ("conv", "small", "7s2", 64, 64), ("conv", "batch2", "5s2", 32, 32),
    ("conv", "zc96", "zc", 32, 64), ("conv", "zc128", "zc", 64, 64), ("conv", "zc512", "zc", 32, 32),
    ("deconv", "small", "5s2", 64, 32), ("deconv", "small", "5s5", 32, 64), ("deconv", "zc128", "zc", 64, 64),
    ("deconv", "zc512", "zc", 32, 64),
]


def _winputs(case, seed=0):
    kind, level, shape, cin, cout = case
    rs = np.random.RandomState(seed + 7 * cin + 13 * cout + sum(map(ord, kind + level + shape)))
    lv = _wlevel(level)
    g = _wgeom(lv, kind, shape)
    x = tx.grid_x(rs, g["n_src"], cin)
    w = tx.grid_w(rs, g["K"], cin, cout)
    dy = tx.grid_w(rs, g["n_dst"], cout)
    return lv, g, x, w, dy


@pytest.mark.gpu
@pytest.mark.parametrize("case", EXACT_CASES, ids=tx._cid)
@pytest.mark.parametrize("mode", list(tx.MODES))
def test_exact_grid_bitwise_wide(mode, case):
    """Forward, input gradient and weight gradient equal the fp64 reference bit for bit.  In the tensor-core modes every
    forward of a K > 64 plan runs ceil(K / 63) chunked launches and no CUDA-core launch."""
    if mode != "fp32":
        tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv, g, x, w, dy = _winputs(case)
    want = tx.ref_forward(lv, kind, g, x, w)
    try:
        tx._set_mode(mode)
        before = _counters()
        out, _ = tx.run_forward(lv, kind, g, x, w)
        d = _delta(before)
        print(f"[wide] {mode} {tx._cid(case)} forward: {d}")
        tx.assert_exact(out, want, f"{mode} {tx._cid(case)} forward")
        tc, chunk = _forward_on_tc(mode, kind, g, cout, g["n_src"])
        assert d["tc"] == tc and d["chunk"] == chunk and d["simt"] == int(tc == 0), d
        before = _counters()
        d_in, dw = tx.run_backward(lv, kind, g, x, dy, w)
        d = _delta(before)
        print(f"[wide] {mode} {tx._cid(case)} backward: {d}")
        want_din, want_dw = tx.ref_backward(lv, kind, g, x, dy, w)
        tx.assert_exact(d_in, want_din, f"{mode} {tx._cid(case)} input gradient")
        tx.assert_exact(dw, want_dw, f"{mode} {tx._cid(case)} weight gradient")
        odd = all(v % 2 for v in g["f"])
        if mode != "fp32" and cin % 32 == 0 and ((kind == "subm" and odd) or kind == "deconv"):
            assert d["chunk"] == _chunks(g["K"]), d  # input gradient: the reversed-offset plan / the strided plan, chunked
    finally:
        tx._set_mode("fp32")


# ------------------------------------------------------------------ GPU: fused epilogue across chunks
EPI_CASES = [(("subm", "small", "5", 64, 64), True, True), (("subm", "mini4", "7", 32, 128), True, False),
             (("conv", "zc128", "zc", 64, 64), False, True), (("conv", "small", "5s2", 32, 32), True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("case,bias,addend", EPI_CASES, ids=lambda v: tx._cid(v) if isinstance(v, tuple) else str(v))
@pytest.mark.parametrize("mode", tx.TC_MODES)
def test_fused_epilogue_across_chunks_exact(mode, case, bias, addend):
    """Bias and the caller's addend go into the first chunk, the bf16 copy into the last: out equals the fp64 reference and the
    bf16 copy equals out.to(bfloat16); rows beyond the output stay untouched (run_forward's sentinel tail)."""
    tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv, g, x, w, _ = _winputs(case, seed=1)
    rs = np.random.RandomState(cin + cout)
    b = tx.grid_w(rs, cout) if bias else None
    ad = tx.grid_w(rs, g["n_dst"], cout) if addend else None
    want = tx.ref_forward(lv, kind, g, x, w, b, ad)
    try:
        tx._set_mode(mode)
        before = _counters()
        out, o16 = tx.run_forward(lv, kind, g, x, w, b, ad, want16=True)
        d = _delta(before)
    finally:
        tx._set_mode("fp32")
    print(f"[wide epilogue] {mode} {tx._cid(case)} bias={bias} add={addend}: {d}")
    assert d["chunk"] == _chunks(g["K"]) and d["simt"] == 0, d
    tx.assert_exact(out, want, f"{mode} {tx._cid(case)} epilogue")
    assert torch.equal(o16.view(torch.int16), out.to(torch.bfloat16).view(torch.int16)), "bf16 copy differs from out.to(bfloat16)"


@pytest.mark.gpu
@pytest.mark.parametrize("kind,level,shape", [("deconv", "small", "5s5"), ("deconv", "zc128", "zc"), ("subm", "mini4", "5"), ("subm", "small", "5")])
@pytest.mark.parametrize("mode", tx.TC_MODES)
def test_lateral_stage_and_epilogue_stats_wide(mode, kind, level, shape):
    """out = conv(x) + y[row] @ W_lat with the epilogue statistics of out, in one launch.  Deconvolutions with one parent per fine
    site (K = 125: 5^3 / 5; K = 128: the z-collapse) run per-tile weight slices; on 5^3 submanifold plans the lateral stage and the
    statistics go into the last chunk (the small building splits its offsets over CTAs: no statistics there)."""
    tx._tc_or_skip()
    lv = _wlevel(level)
    g = _wgeom(lv, kind, shape)
    C0, n, c_lat = 64, g["n_dst"], 32
    rs = np.random.RandomState(g["K"])
    x, w = tx.grid_x(rs, g["n_src"], C0, 0.1), tx.grid_w(rs, g["K"], C0, C0)
    y, wl = tx.grid_x(rs, n, c_lat, 0.1), tx.grid_w(rs, c_lat, C0)
    want = tx.ref_forward(lv, kind, g, x, w) + y.double() @ wl.double()
    s1, s2 = want.sum(0), (want * want).sum(0)
    lib = tx._lib()
    import ctypes as C
    try:
        tx._set_mode(mode)
        stats = torch.zeros(8 * 2 * 128, dtype=torch.float64, device="cuda")
        y16 = y.to(torch.bfloat16)
        before = _counters()
        tx._check(lib.scn_fuse_next_lateral(tx._p(y), tx._p(y16), tx._p(wl), 0, c_lat, n))
        tx._check(lib.scn_fuse_next_stats(tx._p(stats)))
        out, _ = tx.run_forward(lv, kind, g, x, w)
        took_l, took_s = C.c_int(), C.c_int()
        tx._check(lib.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
        d = _delta(before)
    finally:
        tx._set_mode("fp32")
    print(f"[wide lateral] {mode} {kind} {level}: {d}, stats taken {took_s.value}")
    assert took_l.value == 1 and d["lateral"] == 1, d
    if kind == "subm":
        assert d["chunk"] == _chunks(g["K"]), d
    tx.assert_exact(out, want, f"{mode} {kind} {level} lateral")
    if d["split"] == 0:
        assert took_s.value == 1 and d["stats"] == 1, d
        got1, got2 = tx._stats_sums(stats, C0)
        tx.assert_exact(got1, s1, "epilogue sum")
        tx.assert_exact(got2, s2, "epilogue sum of squares")
    else:
        assert took_s.value == 0


# ------------------------------------------------------------------ GPU: per layer against the oracle on N(0, 1) data
@pytest.mark.gpu
@pytest.mark.parametrize("case", [("subm", "mini4", "5", 64, 64), ("subm", "small", "7", 32, 64), ("conv", "small", "5s2", 64, 128),
                                  ("conv", "zc128", "zc", 64, 64), ("deconv", "zc512", "zc", 64, 32)], ids=tx._cid)
@pytest.mark.parametrize("mode", list(tx.MODES))
def test_layer_tolerance_random(mode, case):
    if mode != "fp32":
        tx._tc_or_skip()
    kind, level, shape, cin, cout = case
    lv = _wlevel(level)
    g = _wgeom(lv, kind, shape)
    gen = torch.Generator(device="cuda").manual_seed(cin + cout)
    x = torch.randn(g["n_src"], cin, device="cuda", generator=gen)
    w = torch.randn(g["K"], cin, cout, device="cuda", generator=gen) / np.sqrt(cin * g["K"])
    want = tx.ref_forward(lv, kind, g, x, w)
    try:
        tx._set_mode(mode)
        out, _ = tx.run_forward(lv, kind, g, x, w)
    finally:
        tx._set_mode("fp32")
    rtol, atol = LAYER_TOL[mode]
    err = (out.double() - want).abs()
    bound = rtol * want.abs() + atol * float(want.abs().max())
    print(f"[wide tol] {mode} {tx._cid(case)}: max err {float(err.max()):.3e} of max|ref| {float(want.abs().max()):.3e}")
    assert bool((err <= bound).all()), float((err - bound).max())


# ------------------------------------------------------------------ GPU: deterministic mode
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(tx.MODES))
def test_deterministic_mode_wide(mode):
    """Bitwise repeats of forward and backward with zero float-atomic launches, on a level whose offsets are split over CTAs."""
    if mode != "fp32":
        tx._tc_or_skip()
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        tx._set_mode(mode)
        for case in (("subm", "small", "5", 64, 64), ("conv", "small", "7s2", 32, 64), ("deconv", "zc128", "zc", 64, 64)):
            kind = case[0]
            rs = np.random.RandomState(3)
            lv, g, _, _, _ = _winputs(case)
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
            assert d["atomic"] == 0, (case, d)
            for a, b in zip(*runs):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), case
    finally:
        tx._set_mode("fp32")
        torch.use_deterministic_algorithms(on, warn_only=warn)


# ------------------------------------------------------------------ GPU: FPN_Net end to end
def _wide_fpn_config():
    """mini4 with 5^3 / 2 downsampling into levels 1 and 2 (levels [73, 73, 521] -> [35, 35, 259] -> [16, 16, 128] -> [8, 8, 64]:
    (n - 1) * 2 + 5 = the finer size) and RPN maps on levels 2 and 1, whose z-collapse filters are [1, 1, 128] and [1, 1, 259]."""
    cfg = fpn_util.mini4_config()
    cfg.update(full_scale=[73, 73, 521], downsample=[[[5, 5, 5], [5, 5, 5], [2, 2, 2]], [[2, 2, 2]] * 3], fpn_scales_from_top=[1, 2],
               rpn_map_sizes=[[16, 16, 128], [35, 35, 259]])
    return cfg


FPN_BLD = dict(nx=60, ny=56, nz=60, n_walls=3, seed=3)
FPN_SIZES = [[73, 73, 521], [35, 35, 259], [16, 16, 128], [8, 8, 64]]  # the port assumes full // 2^level: given explicitly here


def _fpn_inputs():
    coords = synthetic.building_coords(**FPN_BLD)
    return coords, fpn_util.features_for(coords)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(tx.MODES))
def test_fpn_wide_filters_end_to_end(mode, monkeypatch):
    """Recording forward and two replays against the oracle port."""
    if mode != "fp32":
        tx._tc_or_skip()
    import detection_3d_b200.sparseconvnet as scn
    from oracle import fpn_oracle
    monkeypatch.setattr(fpn_oracle, "_sizes", lambda full, n: [list(v) for v in FPN_SIZES[:n]])
    cfg = _wide_fpn_config()
    net = scn.FPN_Net(**cfg)
    state = fpn_util.deterministic_state(net, seed=1)
    net.load_state_dict(state)
    net = net.cuda().eval()
    coords, feats = _fpn_inputs()
    orpn, oroi, _ = fpn_oracle.run_fpn_port(cfg, state, coords, feats)
    # end to end: fp32 / tf32x3 as test_gpu_tf32x3.py, tf32 / bf16 as smoke() (max error over max|ref|)
    rtol, atol = {"fp32": (2e-3, 2e-4), "tf32x3": (2e-3, 2e-4), "tf32": (0, 3e-2), "bf16": (0, 6e-2)}[mode]
    try:
        scn.set_math_mode(mode)
        before = _counters()
        for rep in range(3):  # records, then replays
            with torch.no_grad():
                rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats).cuda()])
            torch.cuda.synchronize()
            for a, b in zip(rpn + roi, orpn + oroi):
                assert np.array_equal(a.get_spatial_locations().numpy(), b["locations"]), rep
                ref = b["features"]
                got = a.features.cpu().numpy()
                np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol * max(1.0, float(np.abs(ref).max())), err_msg=f"pass {rep}")
        d = _delta(before)
        print(f"[wide fpn] {mode}: {d}")
        assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
        if mode != "fp32":
            assert d["chunk"] > 0, d
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.gpu
def test_fpn_wide_filters_replayed_training_step():
    """The replayed training step (scn_program_run in training mode + scn_program_backward) in tf32x3 mode against the
    layer-by-layer fp32-mode step of the same network: loss, every parameter gradient within the fp32-mode bounds of
    test_gpu_tf32x3.test_training_step_vs_reference_autograd."""
    tx._tc_or_skip()
    import detection_3d_b200.sparseconvnet as scn
    cfg = dict(_wide_fpn_config(), track_running_stats=True)
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
        scn.set_math_mode("tf32x3")
        net = scn.FPN_Net(**cfg).cuda().train()
        step(net)  # records the training program
        assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")
        before = _counters()
        loss, g = step(net)
        d = _delta(before)
    finally:
        scn.set_math_mode("fp32")
    print(f"[wide train] {d}")
    assert d["train_replay"] == 1 and d["chunk"] > 0 and d["x3"] > 0, d
    assert abs(loss - loss32) <= 5e-3 * loss32
    assert set(g) == set(g32)
    worst = 0.0
    for k in g32:
        err = float((g[k] - g32[k]).abs().max() / max(1e-6, float(g32[k].abs().max())))
        worst = max(worst, err)
        assert err < 5e-3, (k, err)
    print(f"[wide train] worst gradient error {worst:.3e} of max|grad|")
