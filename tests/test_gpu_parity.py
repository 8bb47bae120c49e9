"""GPU parity tests (run on the B200 box): every result of the CUDA path, obtained through the
C-ABI, against the CPU oracle on the same seeded inputs, against the committed golden vectors
generated from the reference itself, and -- at BASELINE.json's full size -- by digest."""
import json
import os

import numpy as np
import pytest
import torch

import fpn_util
from detection_3d_b200 import synthetic
from oracle import fpn_oracle
from oracle import scn_oracle as so

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _gpu():
    from gpu_adapter import GpuMetadata
    return GpuMetadata()


def _cat_iter(md, sz):
    return np.concatenate([md.iteration_order(sz, b) for b in range(md.batch_size(sz))] or [np.zeros(0, np.int32)])


def _compare_metadata(G, O, full, n_levels, pro=(), extra_convs=()):
    for a, b in zip(G.input_rules(), O.input_rules()):
        assert np.array_equal(a, b), "input rules"
    sizes = fpn_util.pyramid_sizes(full, n_levels)
    for l, sz in enumerate(sizes):
        assert G.nactive(sz) == O.nactive(sz), f"nActive level {l}"
        assert np.array_equal(G.spatial_locations(sz), O.spatial_locations(sz)), f"locations level {l}"
        gi, oi = _cat_iter(G, sz), _cat_iter(O, sz)
        assert np.array_equal(gi, oi), f"hash-iteration order level {l}: first diff at {int(np.argmax(gi != oi)) if gi.shape == oi.shape else 'shape'}"
        for k, (a, b) in enumerate(zip(G.submanifold_rules(sz, [3, 3, 3]), O.submanifold_rules(sz, [3, 3, 3]))):
            assert np.array_equal(a, b), f"submanifold rules level {l} offset {k}"
        if l + 1 < n_levels:
            for k, (a, b) in enumerate(zip(G.conv_rules(sz, sizes[l + 1], [2, 2, 2], [2, 2, 2]), O.conv_rules(sz, sizes[l + 1], [2, 2, 2], [2, 2, 2]))):
                assert np.array_equal(a, b), f"conv rules level {l} offset {k}"
    for l in pro:
        sz = sizes[l]
        o = [sz[0], sz[1], 1]
        for k, (a, b) in enumerate(zip(G.conv_rules(sz, o, [1, 1, sz[2]], [1, 1, 1]), O.conv_rules(sz, o, [1, 1, sz[2]], [1, 1, 1]))):
            assert np.array_equal(a, b), f"pro2d rules level {l} offset {k}"
        assert np.array_equal(G.spatial_locations(o), O.spatial_locations(o))


# ------------------------------------------------------------------ rulebooks (bit exact)
def test_small_rulebook_golden():
    g = np.load(os.path.join(GOLD, "rulebook_small.npz"))
    G = _gpu()
    assert G.input_layer([8, 8, 8], g["coords"][:, :3], 0, 4) == 6
    hdr, tab = G.input_rules()
    assert hdr.tolist() == [4, 2, 7, 6] and np.array_equal(tab, g["input1"])
    assert np.array_equal(G.iteration_order([8, 8, 8]), g["iter"])
    for k, r in enumerate(G.submanifold_rules([8, 8, 8], [3, 3, 3])):
        assert np.array_equal(r, g[f"subm{k}"]), k
    for k, r in enumerate(G.conv_rules([8, 8, 8], [4, 4, 4], [2, 2, 2], [2, 2, 2])):
        assert np.array_equal(r, g[f"conv{k}"]), k
    assert np.array_equal(G.spatial_locations([4, 4, 4]), g["loc4"])
    for k, r in enumerate(G.conv_rules([4, 4, 4], [4, 4, 1], [1, 1, 4], [1, 1, 1])):
        assert np.array_equal(r, g[f"pro{k}"]), k


@pytest.mark.parametrize("case", ["building", "random_dense", "random_sparse", "single_point", "line", "big_coords", "dev_coords"])
def test_rulebooks_vs_oracle(case):
    rs = np.random.RandomState(7)
    full, nl, pro = [64, 64, 32], 4, (1, 2)
    if case == "building":
        c = synthetic.small_building(40, 36, 12, 3, seed=1)
    elif case == "random_dense":
        c = rs.randint(0, 24, (20000, 3))
    elif case == "random_sparse":
        c = np.stack([rs.randint(0, 64, 3000), rs.randint(0, 64, 3000), rs.randint(0, 32, 3000)], 1)
    elif case == "single_point":
        c = np.array([[5, 6, 7]])
    elif case == "line":
        c = np.stack([np.arange(64), np.full(64, 3), np.full(64, 31)], 1)
    elif case == "big_coords":
        full, nl, pro = [2048, 2048, 512], 9, (4, 5)
        c = np.stack([rs.randint(1500, 2048, 30000), rs.randint(0, 2048, 30000), rs.randint(400, 512, 30000)], 1)
    else:
        c = synthetic.small_building(50, 30, 20, 4, seed=2)
    G, O = _gpu(), so.OracleMetadata()
    n = G.input_layer(full, c, 0, 4, coords_on_device=(case == "dev_coords"))
    assert n == O.input_layer(full, c, 0, 4)
    _compare_metadata(G, O, full, nl, pro)


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_input_layer_modes_and_features(mode):
    rs = np.random.RandomState(mode)
    c = rs.randint(0, 12, (3000, 3))
    if mode == 0:
        c = np.unique(c, axis=0)
        c = c[rs.permutation(c.shape[0])]
    f = rs.randn(c.shape[0], 9).astype(np.float32)
    G, O = _gpu(), so.OracleMetadata()
    assert G.input_layer([16, 16, 16], c, 0, mode, feats=f) == O.input_layer([16, 16, 16], c, 0, mode)
    assert np.array_equal(G.spatial_locations([16, 16, 16]), O.spatial_locations([16, 16, 16]))
    if mode == 0:
        want = f
    else:
        for a, b in zip(G.input_rules(), O.input_rules()):
            assert np.array_equal(a, b)
        hdr, tab = O.input_rules()
        if mode in (1, 2):
            want = f[tab.reshape(-1, 2)[:, 1]]
        else:
            want = so.o_input_layer_forward(f, hdr, tab)
    np.testing.assert_allclose(G.input_features.cpu().numpy(), want, rtol=1e-6, atol=1e-6)


def test_batched_input_with_batch_size_hint():
    rs = np.random.RandomState(3)
    c = np.concatenate([rs.randint(0, 20, (6000, 3)), rs.randint(0, 3, (6000, 1))], 1)  # interleaved batch items
    G, O = _gpu(), so.OracleMetadata()
    assert G.input_layer([32, 32, 32], c, 3, 4) == O.input_layer([32, 32, 32], c, 3, 4)
    _compare_metadata(G, O, [32, 32, 32], 3, (1,))


def test_empty_input():
    G = _gpu()
    assert G.input_layer([16, 16, 16], np.zeros((0, 4), np.int64), 0, 4) == 0
    assert G.spatial_locations([16, 16, 16]).shape == (0, 4)
    assert all(r.shape[0] == 0 for r in G.submanifold_rules([16, 16, 16], [3, 3, 3]))


@pytest.mark.parametrize("f,s", [([3, 3, 3], [2, 2, 2]), ([4, 4, 4], [2, 2, 2]), ([3, 1, 2], [2, 1, 2]), ([2, 2, 2], [2, 2, 2])])
def test_overlapping_strided_rulebooks(f, s):
    rs = np.random.RandomState(11)
    full = [33, 33, 34] if f[0] == 3 else [32, 32, 32]
    if f == [3, 1, 2]:
        full = [33, 20, 32]
    c = np.stack([rs.randint(0, full[d], 5000) for d in range(3)], 1)
    out = [(full[d] - f[d]) // s[d] + 1 for d in range(3)]
    G, O = _gpu(), so.OracleMetadata()
    assert G.input_layer(full, c, 0, 4) == O.input_layer(full, c, 0, 4)
    for k, (a, b) in enumerate(zip(G.conv_rules(full, out, f, s), O.conv_rules(full, out, f, s))):
        assert np.array_equal(a, b), k
    assert np.array_equal(G.spatial_locations(out), O.spatial_locations(out))


@pytest.mark.parametrize("name,bld,full,nl,pro", [
    ("mini4", dict(nx=60, ny=56, nz=24, n_walls=3, seed=3), [64, 64, 32], 4, (1, 2)),
    ("sw4c_mid", dict(nx=300, ny=280, nz=40, n_walls=5, seed=5), [2048, 2048, 512], 9, (4, 5, 6)),
    ("b470", dict(), [2048, 2048, 512], 9, (4, 5, 6)),
])
def test_rulebook_digests_vs_reference_golden(name, bld, full, nl, pro):
    """Full-size check by checksum of checksums against digests taken from the reference's own
    Metadata<3> (tests/golden/rulebooks.json)."""
    gold = json.load(open(os.path.join(GOLD, "rulebooks.json")))[name]
    coords = synthetic.building_coords(**bld)
    G = _gpu()
    G.input_layer(full, coords, 0, 4)
    got = fpn_util.metadata_digests(G, full, nl, pro)
    got["input_rules"] = fpn_util.rulebook_digest(G.input_rules())
    got["n_input_rows"] = int(coords.shape[0])
    bad = {k: (got.get(k), gold[k]) for k in gold if got.get(k) != gold[k]}
    assert not bad, bad


# ------------------------------------------------------------------ compute kernels
FP32_RTOL, FP32_ATOL = 2e-4, 2e-5   # fp32 CUDA-core path vs fp32 CPU: summation-order noise only


def _close(got, want, rtol=FP32_RTOL, atol=FP32_ATOL):
    want = np.asarray(want)
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    np.testing.assert_allclose(np.asarray(got), want, rtol=rtol, atol=atol * scale)


def _setup_levels():
    import detection_3d_b200.sparseconvnet as scn
    c = synthetic.small_building(40, 36, 12, 3, seed=4)
    G, O = _gpu(), so.OracleMetadata()
    G.input_layer([64, 64, 32], c, 0, 4)
    O.input_layer([64, 64, 32], c, 0, 4)
    return scn, G, O


@pytest.mark.parametrize("cin,cout,f", [(9, 32, 3), (32, 32, 3), (64, 128, 3), (128, 128, 3), (32, 128, 1), (20, 12, 3)])
def test_submanifold_forward_backward(cin, cout, f):
    scn, G, O = _setup_levels()
    scn.set_math_mode("fp32")
    sz = [64, 64, 32]
    n = O.nactive(sz)
    rs = np.random.RandomState(cin * 7 + cout)
    x = rs.randn(n, cin).astype(np.float32)
    w = (rs.randn(f ** 3, 1, cin, cout) * (2.0 / (cin * f ** 3)) ** 0.5).astype(np.float32)
    rules = O.submanifold_rules(sz, [f] * 3)
    want, macs = so.o_conv_forward(x, w, rules, n)
    out = torch.empty(0, device="cuda")
    L = torch.LongTensor
    got_macs = scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([f] * 3), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
    assert got_macs == macs
    _close(out.cpu().numpy(), want)
    dy = rs.randn(n, cout).astype(np.float32)
    din_w, dw_w = so.o_conv_backward(x, dy, w, rules)
    din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
    scn.SCN.SubmanifoldConvolution_backward(L(sz), L([f] * 3), G.m, torch.from_numpy(x).cuda(), din, torch.from_numpy(dy).cuda(),
                                            torch.from_numpy(w).cuda(), dw, torch.Tensor())
    _close(din.cpu().numpy(), din_w)
    _close(dw.cpu().numpy(), dw_w, rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize("cin,cout", [(32, 64), (128, 128)])
def test_strided_conv_and_deconv_forward_backward(cin, cout):
    scn, G, O = _setup_levels()
    scn.set_math_mode("fp32")
    L = torch.LongTensor
    a, b, f, s = [64, 64, 32], [32, 32, 16], [2, 2, 2], [2, 2, 2]
    rules = O.conv_rules(a, b, f, s)
    na, nb = O.nactive(a), O.nactive(b)
    rs = np.random.RandomState(cin + cout)
    x = rs.randn(na, cin).astype(np.float32)
    w = (rs.randn(8, 1, cin, cout) * (2.0 / (cin * 8)) ** 0.5).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, rules, nb)
    out = torch.empty(0, device="cuda")
    got_macs = scn.SCN.Convolution_updateOutput(L(a), L(b), L(f), L(s), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
    assert got_macs == macs and out.shape == (nb, cout)
    _close(out.cpu().numpy(), want)
    dy = rs.randn(nb, cout).astype(np.float32)
    din_w, dw_w = so.o_conv_backward(x, dy, w, rules)
    din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
    scn.SCN.Convolution_backward(L(a), L(b), L(f), L(s), G.m, torch.from_numpy(x).cuda(), din, torch.from_numpy(dy).cuda(), torch.from_numpy(w).cuda(), dw, torch.Tensor())
    _close(din.cpu().numpy(), din_w)
    _close(dw.cpu().numpy(), dw_w, rtol=1e-3, atol=1e-4)
    # deconvolution b -> a reuses the same rulebook reversed
    xc = rs.randn(nb, cin).astype(np.float32)
    want, macs = so.o_conv_forward(xc, w, rules, na, deconv=True)
    out = torch.empty(0, device="cuda")
    got_macs = scn.SCN.Deconvolution_updateOutput(L(b), L(a), L(f), L(s), G.m, torch.from_numpy(xc).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
    assert got_macs == macs and out.shape == (na, cout)
    _close(out.cpu().numpy(), want)
    dy = rs.randn(na, cout).astype(np.float32)
    din_w, dw_w = so.o_conv_backward(xc, dy, w, rules, deconv=True)
    din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
    scn.SCN.Deconvolution_backward(L(b), L(a), L(f), L(s), G.m, torch.from_numpy(xc).cuda(), din, torch.from_numpy(dy).cuda(), torch.from_numpy(w).cuda(), dw, torch.Tensor())
    _close(din.cpu().numpy(), din_w)
    _close(dw.cpu().numpy(), dw_w, rtol=1e-3, atol=1e-4)


def test_z_collapse_convolution():
    scn, G, O = _setup_levels()
    scn.set_math_mode("fp32")
    L = torch.LongTensor
    a, b = [64, 64, 32], [32, 32, 16]
    O.conv_rules(a, b, [2, 2, 2], [2, 2, 2]); G.conv_rules(a, b, [2, 2, 2], [2, 2, 2])
    o, f, s = [32, 32, 1], [1, 1, 16], [1, 1, 1]
    rules = O.conv_rules(b, o, f, s)
    rs = np.random.RandomState(5)
    x = rs.randn(O.nactive(b), 32).astype(np.float32)
    w = (rs.randn(16, 1, 32, 32) * 0.1).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, rules, O.nactive(o))
    out = torch.empty(0, device="cuda")
    got = scn.SCN.Convolution_updateOutput(L(b), L(o), L(f), L(s), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
    assert got == macs
    _close(out.cpu().numpy(), want)


@pytest.mark.parametrize("n,c", [(5000, 32), (777, 128), (3, 256), (2000, 9)])
@pytest.mark.parametrize("mode", ["train", "eval_running", "eval_instance"])
def test_batchnorm_forward_backward(n, c, mode):
    import detection_3d_b200.sparseconvnet as scn
    rs = np.random.RandomState(n + c)
    x = (rs.randn(n, c) * 2 + 0.5).astype(np.float32)
    gam, bet = (1 + 0.1 * rs.randn(c)).astype(np.float32), (0.1 * rs.randn(c)).astype(np.float32)
    rm, rv = (0.1 * rs.randn(c)).astype(np.float32), (1 + 0.2 * rs.rand(c)).astype(np.float32)
    T = lambda a: torch.from_numpy(a.copy()).cuda()
    out, sm, si, trm, trv = torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), T(rm), T(rv)
    if mode == "eval_instance":
        mean = x.mean(0, dtype=np.float64).astype(np.float32)
        var = x.var(0, ddof=1, dtype=np.float64).astype(np.float32)
        want, wsm, wsi = so.o_bn_forward(x, gam, bet, mean, var, 1e-4, 0.9, False, 0.0)
        scn.SCN.BatchNormalization_updateOutput(T(x), out, sm, si, trm, trv, T(gam), T(bet), 1e-4, 0.9, False, 0.0, instance_stats=True)
    else:
        orm, orv = rm.copy(), rv.copy()
        want, wsm, wsi = so.o_bn_forward(x, gam, bet, orm, orv, 1e-4, 0.9, mode == "train", 0.0)
        scn.SCN.BatchNormalization_updateOutput(T(x), out, sm, si, trm, trv, T(gam), T(bet), 1e-4, 0.9, mode == "train", 0.0)
        np.testing.assert_allclose(trm.cpu().numpy(), orm, rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(trv.cpu().numpy(), orv, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(sm.cpu().numpy(), wsm, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(si.cpu().numpy(), wsi, rtol=1e-4, atol=1e-5)
    _close(out.cpu().numpy(), want, rtol=1e-4, atol=1e-5)
    if mode == "train":
        dy = rs.randn(n, c).astype(np.float32)
        din_w, dw_w, db_w = so.o_bn_backward(x, want, dy, wsm, wsi, gam, 0.0)
        din, dw, db = torch.empty(0, device="cuda"), torch.zeros(c, device="cuda"), torch.zeros(c, device="cuda")
        scn.SCN.BatchNormalization_backward(T(x), din, out, T(dy), sm, si, trm, trv, T(gam), T(bet), dw, db, 0.0)
        _close(din.cpu().numpy(), din_w, rtol=1e-3, atol=1e-4)
        _close(dw.cpu().numpy(), dw_w, rtol=1e-3, atol=1e-4)
        _close(db.cpu().numpy(), db_w, rtol=1e-3, atol=1e-4)


# ------------------------------------------------------------------ whole backbone
def _run_product_fpn(cfg, bld, math_mode):
    import detection_3d_b200.sparseconvnet as scn
    scn.set_math_mode(math_mode)
    net = scn.FPN_Net(**cfg)
    state = fpn_util.deterministic_state(net, seed=1)
    net.load_state_dict(state)
    net = net.cuda().eval()
    coords = synthetic.building_coords(**bld)
    feats = fpn_util.features_for(coords)
    scn.forward_pass_multiplyAdd_count = 0
    with torch.no_grad():
        rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats).cuda()])
    torch.cuda.synchronize()
    return rpn, roi, scn.forward_pass_multiplyAdd_count, state, coords, feats


@pytest.mark.parametrize("name,cfgname,bld", [
    ("mini4", "mini4", dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)),
    ("sw4c_mid", "sw4c", dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)),
])
def test_fpn_forward_fp32_vs_reference_golden(name, cfgname, bld):
    """The drop-in FPN_Net on CUDA vs the outputs of the reference's own scn.FPN_Net (golden)."""
    import detection_3d_b200.sparseconvnet as scn
    cfg = fpn_util.mini4_config() if cfgname == "mini4" else scn.sw4c_fpn432_config()
    g = np.load(os.path.join(GOLD, f"fpn_{name}.npz"))
    rpn, roi, macs, *_ = _run_product_fpn(cfg, bld, "fp32")
    assert macs == float(g["macs"])  # same multiply-add counter as the reference
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        assert len(maps) == int(g[f"n_{tag}"])
        for i, m in enumerate(maps):
            assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
            assert m.spatial_size.tolist() == g[f"{tag}{i}_spatial_size"].tolist()
            ref = g[f"{tag}{i}_features"]
            # end-to-end fp32 tolerance after ~40 layers incl. instance-norm on as few as 4 rows
            _close(m.features.cpu().numpy(), ref, rtol=2e-3, atol=2e-4)


def test_fpn_forward_layerwise_vs_oracle():
    """Layer-by-layer taps of the CPU port vs the module outputs (catches compensating errors)."""
    import detection_3d_b200.sparseconvnet as scn
    cfg = fpn_util.mini4_config()
    bld = dict(nx=44, ny=40, nz=20, n_walls=3, seed=9)
    rpn, roi, macs, state, coords, feats = _run_product_fpn(cfg, bld, "fp32")
    orpn, oroi, omacs = fpn_oracle.run_fpn_port(cfg, state, coords, feats)
    assert macs == omacs
    for a, b in zip(rpn + roi, orpn + oroi):
        assert np.array_equal(a.get_spatial_locations().numpy(), b["locations"])
        _close(a.features.cpu().numpy(), b["features"], rtol=2e-3, atol=2e-4)


# ------------------------------------------------------------------ tcgen05 tensor-core path (TF32 inputs, fp32 accumulate)
# TF32 keeps 10 mantissa bits of every operand (activations truncated by the tensor core, weights
# rounded to nearest): per-product relative error <= 2^-10; the tolerance below is that bound
# against the largest output magnitude of the layer.
TF32_RTOL, TF32_ATOL = 4e-3, 2e-3
# BF16 mode ('bf16'): operands (activations AND weights) rounded to nearest bfloat16 (8 mantissa
# bits, relative rounding error <= 2^-9 each), fp32 accumulation in TMEM; layers whose input rows are
# narrower than 64 channels keep TF32 operands.  Per-layer bound = 4x the TF32 one.
BF16_RTOL, BF16_ATOL = 1.6e-2, 8e-3
TC_TOL = {"tf32": (TF32_RTOL, TF32_ATOL), "bf16": (BF16_RTOL, BF16_ATOL)}
TC_E2E = {"tf32": 1e-2, "bf16": 4.5e-2}


def _tc_or_skip(scn):
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")


@pytest.mark.parametrize("math", ["tf32", "bf16"])
@pytest.mark.parametrize("cin,cout,f", [(9, 32, 3), (32, 32, 3), (64, 64, 3), (128, 128, 3), (256, 256, 3), (32, 128, 1), (64, 128, 3), (256, 128, 1), (20, 64, 3),
                                       (48, 256, 3)])  # (48 -> 256: rows padded to 64 channels AND copied to bf16, two scratch buffers in one launch)
def test_tc_submanifold_forward(cin, cout, f, math):
    scn, G, O = _setup_levels()
    _tc_or_skip(scn)
    sz = [64, 64, 32]
    n = O.nactive(sz)
    rs = np.random.RandomState(cin * 3 + cout + f)
    x = rs.randn(n, cin).astype(np.float32)
    w = (rs.randn(f ** 3, 1, cin, cout) * (2.0 / (cin * f ** 3)) ** 0.5).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, O.submanifold_rules(sz, [f] * 3), n)
    L = torch.LongTensor
    try:
        scn.set_math_mode(math)
        out = torch.empty(0, device="cuda")
        got = scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([f] * 3), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert got == macs
    _close(out.cpu().numpy(), want, rtol=TC_TOL[math][0], atol=TC_TOL[math][1])


@pytest.mark.parametrize("math", ["tf32", "bf16"])
def test_tc_input_gradients(math):
    """tf32 / bf16 mode: the input gradient of all three convolution kinds runs on the tcgen05 forward kernel with transposed
    weights (submanifold: symmetric plan with reversed offsets; strided convolution: a deconvolution; deconvolution: the
    strided convolution); d_weight runs on the tcgen05 kernel conv_dw_tc in bf16 mode (every shape here, 9 / 32 / 64 input channels
    included: tests/test_gpu_tc_exact.py reads which kernel ran) and on the fp32 CUDA cores in tf32 mode.  Checked against the
    oracle's backward."""
    scn, G, O = _setup_levels()
    _tc_or_skip(scn)
    L = torch.LongTensor
    T = lambda a: torch.from_numpy(a).cuda()
    rtol, atol = TC_TOL[math]
    try:
        scn.set_math_mode(math)
        sz = [64, 64, 32]
        n = O.nactive(sz)
        for cin, cout, f in [(64, 128, 3), (128, 128, 3), (32, 32, 3), (32, 128, 1), (256, 64, 3), (9, 32, 3)]:
            rs = np.random.RandomState(cin + 3 * cout + f)
            x, dy = rs.randn(n, cin).astype(np.float32), rs.randn(n, cout).astype(np.float32)
            w = (rs.randn(f ** 3, 1, cin, cout) * (2.0 / (cin * f ** 3)) ** 0.5).astype(np.float32)
            rules = O.submanifold_rules(sz, [f] * 3)
            out = torch.empty(0, device="cuda")
            scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([f] * 3), G.m, T(x), out, T(w), torch.Tensor())
            din_w, dw_w = so.o_conv_backward(x, dy, w, rules)
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            scn.SCN.SubmanifoldConvolution_backward(L(sz), L([f] * 3), G.m, T(x), din, T(dy), T(w), dw, torch.Tensor())
            _close(din.cpu().numpy(), din_w, rtol=rtol, atol=atol)
            _close(dw.cpu().numpy(), dw_w, rtol=rtol, atol=atol)
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
            scn.SCN.Convolution_backward(L(a), L(b), L(f), L(s), G.m, T(x), din, T(dy), T(w), dw, torch.Tensor())
            _close(din.cpu().numpy(), din_w, rtol=rtol, atol=atol)
            _close(dw.cpu().numpy(), dw_w, rtol=rtol, atol=atol)
            xc, dyf = rs.randn(nb, cin).astype(np.float32), rs.randn(na, cout).astype(np.float32)
            out = torch.empty(0, device="cuda")
            scn.SCN.Deconvolution_updateOutput(L(b), L(a), L(f), L(s), G.m, T(xc), out, T(w), torch.Tensor())
            din_w, dw_w = so.o_conv_backward(xc, dyf, w, rules, deconv=True)
            din, dw = torch.empty(0, device="cuda"), torch.zeros(w.shape, device="cuda")
            scn.SCN.Deconvolution_backward(L(b), L(a), L(f), L(s), G.m, T(xc), din, T(dyf), T(w), dw, torch.Tensor())
            _close(din.cpu().numpy(), din_w, rtol=rtol, atol=atol)
            _close(dw.cpu().numpy(), dw_w, rtol=rtol, atol=atol)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")


def test_bf16_shadow_from_batchnorm_and_add():
    """In 'bf16' mode BatchNorm / add outputs carry a bfloat16 copy written by the same kernel; the
    convolution that follows gathers from it.  The copy must equal the fp32 output rounded to nearest,
    must be ignored once the tensor was modified in place, and the convolution result must not depend
    on whether the copy or the in-kernel conversion was used."""
    scn, G, O = _setup_levels()
    _tc_or_skip(scn)
    sz = [64, 64, 32]
    n = O.nactive(sz)
    rs = np.random.RandomState(11)
    x = torch.from_numpy(rs.randn(n, 64).astype(np.float32)).cuda()
    w = torch.from_numpy((rs.randn(27, 1, 64, 64) * 0.03).astype(np.float32)).cuda()
    L = torch.LongTensor
    try:
        scn.set_math_mode("bf16")
        y, sm, si = torch.empty(0, device="cuda"), torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        scn.SCN.BatchNormalization_updateOutput(x, y, sm, si, torch.Tensor(), torch.Tensor(), torch.Tensor(), torch.Tensor(), 1e-4, 0.9, False, 0.0, True)
        sh = getattr(y, "_scn_bf16", None)
        assert sh is not None and sh[0].dtype == torch.bfloat16
        assert torch.equal(sh[0], y.to(torch.bfloat16))
        z = scn.SCN.add_features(y, x)
        assert torch.equal(z._scn_bf16[0], z.to(torch.bfloat16))
        out_a, out_b = torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([3] * 3), G.m, y, out_a, w, torch.Tensor())  # gathers from the shadow
        y2 = y.clone()                                                                                      # no shadow: converted inside the call
        scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([3] * 3), G.m, y2, out_b, w, torch.Tensor())
        # same operands either way; a small level splits the filter offsets over CTAs and sums them with
        # fp32 atomics, so the two runs may differ in the last bits
        assert torch.allclose(out_a, out_b, rtol=1e-5, atol=1e-6)
        y.mul_(2.0)  # in-place edit: the stale shadow must not be used
        assert scn.SCN._shadow_ptr(y) is None
        out_c = torch.empty(0, device="cuda")
        scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([3] * 3), G.m, y, out_c, w, torch.Tensor())
        torch.cuda.synchronize()
        assert torch.allclose(out_c, 2 * out_a, rtol=1e-5, atol=1e-6)
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.parametrize("math", ["tf32", "bf16"])
@pytest.mark.parametrize("cin,cout", [(32, 64), (128, 128), (48, 64)])
def test_tc_strided_conv_and_z_collapse(cin, cout, math):
    scn, G, O = _setup_levels()
    _tc_or_skip(scn)
    L = torch.LongTensor
    a, b, f, s = [64, 64, 32], [32, 32, 16], [2, 2, 2], [2, 2, 2]
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
    try:
        scn.set_math_mode(math)
        out, outz = torch.empty(0, device="cuda"), torch.empty(0, device="cuda")
        scn.SCN.Convolution_updateOutput(L(a), L(b), L(f), L(s), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
        scn.SCN.Convolution_updateOutput(L(b), L(o), L(fz), L([1, 1, 1]), G.m, torch.from_numpy(xz).cuda(), outz, torch.from_numpy(wz).cuda(), torch.Tensor())
        # deconvolution b -> a on the tensor-core path (per-offset tiles of the reversed rulebook)
        xd = rs.randn(O.nactive(b), cin).astype(np.float32)
        wantd, macsd = so.o_conv_forward(xd, w, rules, O.nactive(a), deconv=True)
        outd = torch.empty(0, device="cuda")
        gotd = scn.SCN.Deconvolution_updateOutput(L(b), L(a), L(f), L(s), G.m, torch.from_numpy(xd).cuda(), outd, torch.from_numpy(w).cuda(), torch.Tensor())
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    rt, at = TC_TOL[math]
    _close(out.cpu().numpy(), want, rtol=rt, atol=at)
    _close(outz.cpu().numpy(), wantz, rtol=rt, atol=at)
    assert gotd == macsd and outd.shape == (O.nactive(a), cout)
    _close(outd.cpu().numpy(), wantd, rtol=rt, atol=at)


@pytest.mark.parametrize("math", ["tf32", "bf16"])
def test_tc_large_level_many_supertiles(math):
    """More supertiles than SMs, ragged last tile, on a mid-size building (persistent loop, ring wrap)."""
    import detection_3d_b200.sparseconvnet as scn
    _tc_or_skip(scn)
    c = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
    G, O = _gpu(), so.OracleMetadata()
    full = [2048, 2048, 512]
    n = G.input_layer(full, c, 0, 4)
    assert n == O.input_layer(full, c, 0, 4)
    rs = np.random.RandomState(0)
    x = rs.randn(n, 64).astype(np.float32)
    w = (rs.randn(27, 1, 64, 64) * (2.0 / (64 * 27)) ** 0.5).astype(np.float32)
    want, macs = so.o_conv_forward(x, w, O.submanifold_rules(full, [3, 3, 3]), n)
    L = torch.LongTensor
    try:
        scn.set_math_mode(math)
        out = torch.empty(0, device="cuda")
        got = scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([3, 3, 3]), G.m, torch.from_numpy(x).cuda(), out, torch.from_numpy(w).cuda(), torch.Tensor())
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    assert got == macs
    _close(out.cpu().numpy(), want, rtol=TC_TOL[math][0], atol=TC_TOL[math][1])


@pytest.mark.parametrize("name,cfgname,bld", [
    ("mini4", "mini4", dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)),
    ("sw4c_mid", "sw4c", dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)),
])
@pytest.mark.parametrize("math", ["tf32", "bf16"])
def test_fpn_forward_tensor_core_vs_reference_golden(name, cfgname, bld, math):
    """End-to-end tensor-core backbone vs the reference's fp32 outputs.  Stated tolerance: 1e-2 (TF32)
    / 4.5e-2 (BF16) of the largest magnitude of each returned map (operand rounding through ~40 layers;
    instance norm on as few as 4 rows at the top levels amplifies relative differences).  Measured on
    B200: TF32 <= 5.2e-3, BF16 <= 2.3e-2 (tools/mode_error.py)."""
    import detection_3d_b200.sparseconvnet as scn
    _tc_or_skip(scn)
    cfg = fpn_util.mini4_config() if cfgname == "mini4" else scn.sw4c_fpn432_config()
    g = np.load(os.path.join(GOLD, f"fpn_{name}.npz"))
    try:
        rpn, roi, macs, *_ = _run_product_fpn(cfg, bld, math)
    finally:
        scn.set_math_mode("fp32")
    assert macs == float(g["macs"])
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        for i, m in enumerate(maps):
            assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
            ref = g[f"{tag}{i}_features"]
            got = m.features.cpu().numpy()
            err = np.abs(got - ref).max() / max(1.0, np.abs(ref).max())
            assert err < TC_E2E[math], (tag, i, float(err))


def test_replayed_program_with_internal_numbering_vs_reference_golden():
    """Second forward of the sw4c backbone on the 300x280x40 building = program replay on an internally numbered Metadata
    (rows in spatial order, no hash-order emulation on the critical path; general multi-launch build for the large levels,
    one-launch build for the small ones) with the outputs gathered into the reference numbering: features and row
    coordinates must equal the outputs of the reference's own scn.FPN_Net (golden fixture), like the first forward's."""
    import detection_3d_b200.sparseconvnet as scn
    cfg = scn.sw4c_fpn432_config()
    bld = dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)
    g = np.load(os.path.join(GOLD, "fpn_sw4c_mid.npz"))
    try:
        scn.set_math_mode("fp32")
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().eval()
        coords = synthetic.building_coords(**bld)
        c, f = torch.from_numpy(coords), torch.from_numpy(fpn_util.features_for(coords)).cuda()
        with torch.no_grad():
            net([c, f])  # records
            assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
            for _ in range(2):
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])  # replays
                assert scn.forward_pass_multiplyAdd_count == float(g["macs"])
                for tag, maps in (("rpn", rpn), ("roi", roi)):
                    assert len(maps) == int(g[f"n_{tag}"])
                    for i, m in enumerate(maps):
                        assert np.array_equal(m.get_spatial_locations().numpy(), g[f"{tag}{i}_locations"]), (tag, i)
                        _close(m.features.cpu().numpy(), g[f"{tag}{i}_features"], rtol=2e-3, atol=2e-4)
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")


# ------------------------------------------------------------------ recorded program (one native call per forward)
@pytest.mark.parametrize("math", ["fp32", "bf16"])
def test_recorded_program_matches_layer_by_layer(math):
    """The second and later inference forwards replay the native calls the first one made
    (sparseconvnet/program.py).  Same kernels in the same order: results must agree with the
    layer-by-layer forward to rounding of the atomically accumulated small levels, the row numbering
    exactly, and the multiply-add counter exactly -- also for a DIFFERENT building than the recorded one."""
    import detection_3d_b200.sparseconvnet as scn
    if math != "fp32":
        _tc_or_skip(scn)
    cfg = fpn_util.mini4_config()
    try:
        scn.set_math_mode(math)
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().eval()
        blds = [dict(nx=60, ny=56, nz=24, n_walls=3, seed=3), dict(nx=44, ny=40, nz=20, n_walls=3, seed=9)]
        inputs = []
        for b in blds:
            c = synthetic.building_coords(**b)
            inputs.append((torch.from_numpy(c), torch.from_numpy(fpn_util.features_for(c)).cuda()))
        with torch.no_grad():
            ref = []
            for c, f in inputs:  # layer by layer (a fresh, unrecorded network object shares the weights)
                net.reset_program()
                net.__dict__["_program_error"] = "disabled for the reference run"
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])
                ref.append(([m.features.clone() for m in rpn + roi], [m.get_spatial_locations() for m in rpn + roi], scn.forward_pass_multiplyAdd_count))
            net.reset_program()
            net([inputs[0][0], inputs[0][1]])          # records
            assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
            for (c, f), (feats, locs, macs) in zip(inputs, ref):
                scn.forward_pass_multiplyAdd_count = 0
                rpn, roi = net([c, f])                  # replays
                assert scn.forward_pass_multiplyAdd_count == macs
                for m, fr, lr in zip(rpn + roi, feats, locs):
                    assert torch.equal(m.get_spatial_locations(), lr)
                    assert m.features.shape == fr.shape
                    scale = max(1.0, float(fr.abs().max()))
                    # fp32: only the summation order of the atomically accumulated small levels differs.  bf16: those
                    # last-bit differences flip the bf16 rounding of individual activations of the next layer (one
                    # bf16 ulp = 4e-3 relative), so two runs of the SAME path already differ by ~1e-2 of max|x|.
                    assert float((m.features - fr).abs().max()) <= (1e-4 if math == "fp32" else 4e-2) * scale
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.parametrize("math", ["tf32", "bf16"])
@pytest.mark.parametrize("big", [False, True])
def test_fused_epilogue_add_and_bf16_copy(math, big):
    """scn_submanifold_convolution_forward(..., add_in, out_bf16): out = conv(in) + add_in and the bf16
    copy of the sum, fused into the epilogue.  Checked against the unfused calls (conv, then
    scn_add_features) on a small level (filter offsets split over CTAs, atomic accumulation) and on a
    level with more work items than SMs."""
    import ctypes as C
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200._lib import l3, lib, check
    _tc_or_skip(scn)
    if big:
        c = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
        sz = [2048, 2048, 512]
    else:
        c = synthetic.small_building(40, 36, 12, 3, seed=4)
        sz = [64, 64, 32]
    G = _gpu()
    n = G.input_layer(sz, c, 0, 4)
    rs = np.random.RandomState(7)
    x = torch.from_numpy(rs.randn(n, 64).astype(np.float32)).cuda()
    w = torch.from_numpy((rs.randn(27, 1, 64, 128) * 0.03).astype(np.float32)).cuda()
    r = torch.from_numpy(rs.randn(n, 128).astype(np.float32)).cuda()
    L = torch.LongTensor
    try:
        scn.set_math_mode(math)
        plain = torch.empty(0, device="cuda")
        scn.SCN.SubmanifoldConvolution_updateOutput(L(sz), L([3] * 3), G.m, x, plain, w, torch.Tensor())
        want = scn.SCN.add_features(plain, r)
        fused = torch.empty(n, 128, device="cuda")
        fused16 = torch.empty(n, 128, dtype=torch.bfloat16, device="cuda")
        macs = C.c_double()
        p = lambda t: C.c_void_p(t.data_ptr())
        check(lib().scn_submanifold_convolution_forward(G.m._h, l3(sz), l3([3, 3, 3]), p(x), p(fused), p(w), None, 64, 128, C.byref(macs), None,
                                                        C.c_longlong(0), p(r), p(fused16)))
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")
    scale = max(1.0, float(want.abs().max()))
    assert float((fused - want).abs().max()) <= 1e-5 * scale      # same products; only the order of the atomic sums may differ
    assert torch.equal(fused16, fused.to(torch.bfloat16))


@pytest.mark.gpu
def test_prefetched_metadata_gives_identical_results():
    """FPN_Net.prefetch(coords) builds the next input's Metadata ahead (scn_program_prepare); the forward that follows must
    return exactly what an unprepared forward returns (same kernels, same rulebooks), also when several buildings are
    streamed and a prefetched Metadata goes unused."""
    import torch
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic
    scn.set_math_mode("tf32")
    try:
        cfg = fpn_util.mini4_config()
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=3))
        net = net.cuda().eval()
        builds = []
        for seed, (nx, ny) in enumerate([(44, 40), (36, 48), (52, 33)]):
            c = synthetic.building_coords(nx=nx, ny=ny, nz=20, n_walls=3, seed=seed)
            builds.append((torch.from_numpy(c).cuda(), torch.from_numpy(fpn_util.features_for(c)).cuda()))
        torch.cuda.synchronize()
        with torch.no_grad():
            net(list(builds[0]))  # records the program
            plain = []
            for c, f in builds:
                rpn, roi = net([c, f])
                plain.append([(m.features.clone(), m.get_spatial_locations().clone()) for m in rpn + roi])
            assert net.prefetch(builds[0][0])
            streamed = []
            for i, (c, f) in enumerate(builds):
                rpn, roi = net([c, f])
                if i + 1 < len(builds):
                    net.prefetch(builds[i + 1][0])
                streamed.append([(m.features.clone(), m.get_spatial_locations().clone()) for m in rpn + roi])
            net.prefetch(builds[1][0])       # prefetched but not used by the next forward
            rpn, roi = net(list(builds[2]))
            unused = [(m.features.clone(), m.get_spatial_locations().clone()) for m in rpn + roi]
        torch.cuda.synchronize()
        def same(x, y):  # small levels accumulate split filter offsets atomically: run-to-run differences in the last bits
            (fa, la), (fb, lb) = x, y
            assert torch.equal(la, lb)
            assert float((fa - fb).abs().max()) <= 1e-3 * max(1.0, float(fa.abs().max()))
        for a, b in zip(plain, streamed):
            for x, y in zip(a, b):
                same(x, y)
        for x, y in zip(plain[2], unused):
            same(x, y)
    finally:
        scn.set_math_mode("fp32")
