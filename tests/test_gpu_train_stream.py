"""Streamed training steps: FPN_Net.prefetch(coords) in train mode prepares the next replayed training step
(scn_program_prepare_training) -- its internally numbered Metadata, the reference-numbered twin on the caller's Metadata, its
plans and the rule lists its backward pass reads -- while the current step runs.

A prefetched step must compute exactly what an unprefetched one computes: same Metadata kind, same kernels, so under
torch.use_deterministic_algorithms(True) every output map, loss term, gradient and BatchNorm running statistic is equal bit for
bit (the BatchNorm saveMean / saveInvStd of a replayed step stay inside the native program; they enter the running statistics and
every gradient).  scn_debug_counter(20) counts training runs that took a prepared Metadata, scn_debug_counter(19) rule lists a
backward entry found already built by a prefetch worker (only prepared steps hint them; unprepared steps build them on demand)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fpn_util
from gpu_adapter import GpuMetadata
from detection_3d_b200 import synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RULES_AHEAD, TRAIN_PREPARED, CHUNKS = 19, 20, 0

# two buildings per network: A, B, A
CASES = {
    "mini4": (lambda scn: fpn_util.mini4_config(), [dict(nx=60, ny=56, nz=24, n_walls=3, seed=3), dict(nx=44, ny=40, nz=20, n_walls=3, seed=9)],
              ([64, 64, 32], 4, (1, 2))),
    "sw4c": (lambda scn: scn.sw4c_fpn432_config(), [dict(nx=300, ny=280, nz=40, n_walls=5, seed=5), dict(nx=260, ny=300, nz=36, n_walls=4, seed=6)],
             ([2048, 2048, 512], 9, (4, 5, 6))),
}


class ReturnedMetadata(GpuMetadata):
    """The adapter over the caller's Metadata a training step returned with its maps."""

    def __init__(self, m):
        self.m = m


@pytest.fixture
def det():
    on, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn)


def _scn(math):
    import detection_3d_b200.sparseconvnet as scn
    if not scn.SCN.lib().scn_tensor_core_path_available():
        pytest.skip("tcgen05 path needs an sm_100 device")
    scn.set_math_mode(math)
    return scn


def _count(i):
    from detection_3d_b200._lib import lib
    return lib().scn_debug_counter(i)


def _net(scn, case):
    cfg = dict(CASES[case][0](scn), track_running_stats=True)
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    return net.cuda().train()


def _inputs(bld, batch_items=1, device="cuda"):
    cs = [synthetic.building_coords(**dict(bld, batch_index=b, seed=bld["seed"] + b)) for b in range(batch_items)]
    c = np.concatenate(cs)
    return torch.from_numpy(c).to(device), torch.from_numpy(fpn_util.features_for(c)).cuda()


def _record(net, inputs):
    """the first training step runs layer by layer and records the program"""
    assert not net.prefetch(inputs[0]), "prefetch before the training program is recorded"
    rpn, roi = net(list(inputs))
    sum((m.features ** 2).mean() for m in rpn + roi).backward()
    torch.cuda.synchronize()
    assert net.__dict__.get("_program_train") is not None, net.__dict__.get("_program_train_error")


def _steps(net, seq, prefetch):
    """training steps on the inputs `seq` (parameters reset before each); with `prefetch`, step i+1 is prepared before step i's
    forward runs (the first) or before its backward (the rest).  -> per step: (maps, loss terms, gradients, buffers); the last
    step's maps"""
    state = {k: v.clone() for k, v in net.state_dict().items()}
    out, last = [], None
    if prefetch:
        assert net.prefetch(seq[0][0])
    for i, (c, f) in enumerate(seq):
        net.load_state_dict(state)
        net.zero_grad(set_to_none=True)
        rpn, roi = net([c, f])
        maps = rpn + roi
        if prefetch and i + 1 < len(seq):
            assert net.prefetch(seq[i + 1][0])  # before backward() of step i: step i's activations and Metadata stay untouched
        terms = [(m.features ** 2).mean() for m in maps]
        sum(terms).backward()
        torch.cuda.synchronize()
        out.append(([m.features.detach().clone() for m in maps], torch.stack([t.detach() for t in terms]),
                    {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None},
                    {k: b.clone() for k, b in net.named_buffers()}))
        last = maps
    return out, last


def _same(a, b):
    for (ma, ta, ga, ba), (mb, tb, gb, bb) in zip(a, b):
        assert len(ma) == len(mb)
        for i, (x, y) in enumerate(zip(ma, mb)):
            assert x.shape == y.shape and torch.equal(x, y), ("map", i)
        assert torch.equal(ta, tb)
        assert ga.keys() == gb.keys()
        for k in ga:
            assert torch.equal(ga[k], gb[k]), k
        for k in ba:
            assert torch.equal(ba[k], bb[k]), k


def test_prefetch_is_used_and_finds_rule_lists_built():
    """prefetch returns False until the training program is recorded; a prepared step takes its Metadata (counter 20) and its
    backward pass finds rule lists built ahead (counter 19); an unprepared step builds its lists on demand"""
    scn = _scn("bf16")
    try:
        net = _net(scn, "mini4")
        a, b = (_inputs(bld) for bld in CASES["mini4"][1])
        _record(net, a)
        assert net.prefetch(b[0])
        p0, r0 = _count(TRAIN_PREPARED), _count(RULES_AHEAD)
        rpn, roi = net(list(a))  # another tensor: the entry for b stays
        sum((m.features ** 2).mean() for m in rpn + roi).backward()
        torch.cuda.synchronize()
        assert _count(TRAIN_PREPARED) == p0
        assert _count(RULES_AHEAD) == r0, "an unprepared step found rule lists built ahead"
        rpn, roi = net(list(b))
        sum((m.features ** 2).mean() for m in rpn + roi).backward()
        torch.cuda.synchronize()
        assert _count(TRAIN_PREPARED) == p0 + 1
        assert _count(RULES_AHEAD) > r0, "the backward pass built every rule list itself"
    finally:
        scn.set_math_mode("fp32")


@pytest.mark.parametrize("math", ["bf16", "tf32x3"])
@pytest.mark.parametrize("case", ["mini4", "sw4c"])
def test_prefetched_steps_bitwise_equal(det, case, math):
    """steps on buildings A, B, A with prefetch one step ahead (step i+1 prepared before step i's backward) equal the same steps
    without prefetch bit for bit; the caller's Metadata of the last step (locations, iteration orders, submanifold and strided
    rulebooks of the twin) equals the unprefetched step's"""
    scn = _scn(math)
    try:
        nets = [_net(scn, case), _net(scn, case)]
        a, b = (_inputs(bld) for bld in CASES[case][1])
        for net in nets:
            _record(net, a)
        seq = [a, b, a]
        p0 = _count(TRAIN_PREPARED)
        plain, md_plain = _steps(nets[0], seq, prefetch=False)
        assert _count(TRAIN_PREPARED) == p0
        streamed, md_streamed = _steps(nets[1], seq, prefetch=True)
        assert _count(TRAIN_PREPARED) == p0 + len(seq)
        _same(plain, streamed)
        for x, y in zip(md_plain, md_streamed):
            assert torch.equal(x.get_spatial_locations(), y.get_spatial_locations())
        if math == "bf16":
            full, nl, pro = CASES[case][2]
            dp = fpn_util.metadata_digests(ReturnedMetadata(md_plain[0].metadata), full, nl, pro)
            ds = fpn_util.metadata_digests(ReturnedMetadata(md_streamed[0].metadata), full, nl, pro)
            assert dp == ds
    finally:
        scn.set_math_mode("fp32")


def _compare(batch_items, device):
    """A, B, A with and without prefetch, bit for bit (mini4, bf16, deterministic)"""
    scn = _scn("bf16")
    torch.use_deterministic_algorithms(True)
    try:
        nets = [_net(scn, "mini4"), _net(scn, "mini4")]
        a, b = (_inputs(bld, batch_items, device) for bld in CASES["mini4"][1])
        for net in nets:
            _record(net, a)
        p0 = _count(TRAIN_PREPARED)
        plain, _ = _steps(nets[0], [a, b, a], prefetch=False)
        streamed, _ = _steps(nets[1], [a, b, a], prefetch=True)
        assert _count(TRAIN_PREPARED) == p0 + 3
        _same(plain, streamed)
    finally:
        torch.use_deterministic_algorithms(False)
        scn.set_math_mode("fp32")


def test_rule_lists_ahead_equal_on_demand(det, monkeypatch):
    """prefetched steps with the rule lists built ahead equal prefetched steps whose backward pass builds them itself
    (SCN_TRAIN_LISTS_AHEAD=0, read at every prepare), bit for bit"""
    scn = _scn("bf16")
    try:
        nets = [_net(scn, "sw4c"), _net(scn, "sw4c")]
        a, b = (_inputs(bld) for bld in CASES["sw4c"][1])
        for net in nets:
            _record(net, a)
        r0 = _count(RULES_AHEAD)
        ahead, _ = _steps(nets[0], [a, b, a], prefetch=True)
        r1 = _count(RULES_AHEAD)
        assert r1 > r0
        monkeypatch.setenv("SCN_TRAIN_LISTS_AHEAD", "0")
        on_demand, _ = _steps(nets[1], [a, b, a], prefetch=True)
        assert _count(RULES_AHEAD) == r1
        _same(ahead, on_demand)
    finally:
        scn.set_math_mode("fp32")


def test_prefetch_two_batch_items_host_coordinates():
    """two batch items: the step runs on the caller's Metadata, prepared with scn_program_prepare; coordinates on the host"""
    _compare(2, "cpu")


def test_prefetch_without_internal_numbering():
    """SCN_TRAIN_INTERNAL=0 (read once per process): training steps run on the caller's Metadata, prepared with
    scn_program_prepare"""
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_train_stream as t; t._compare(1, 'cuda')" % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SCN_TRAIN_INTERNAL="0"), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_prefetched_entry_ignored(det):
    """an entry is not used by a forward of another tensor with the same values, of coordinates modified in place after prefetch,
    in another math mode, or in eval mode; inference prefetches are never used by training; results stay those of an
    unprefetched step"""
    scn = _scn("bf16")
    try:
        net, ref = _net(scn, "mini4"), _net(scn, "mini4")
        a, b = (_inputs(bld) for bld in CASES["mini4"][1])
        _record(net, a)
        _record(ref, a)
        state = {k: v.clone() for k, v in net.state_dict().items()}
        want, _ = _steps(ref, [b], prefetch=False)
        p0 = _count(TRAIN_PREPARED)

        assert net.prefetch(b[0])
        got, _ = _steps(net, [(b[0].clone(), b[1])], prefetch=False)  # another tensor
        _same(want, got)
        c = b[0].clone()
        assert net.prefetch(c)
        c[0, 0] = c[0, 0]  # modified in place (same values, new version)
        net.load_state_dict(state)  # (every step updates the running statistics)
        got, _ = _steps(net, [(c, b[1])], prefetch=False)
        _same(want, got)
        assert _count(TRAIN_PREPARED) == p0

        assert net.prefetch(b[0])
        scn.set_math_mode("tf32")
        assert not net.prefetch(b[0]), "prefetch in a math mode the program was not recorded in"
        rpn, roi = net(list(b))  # layer by layer in tf32 mode
        sum((m.features ** 2).mean() for m in rpn + roi).backward()
        scn.set_math_mode("bf16")
        assert _count(TRAIN_PREPARED) == p0

        assert net.prefetch(b[0])
        net.eval()  # drops the training entries and their memory
        assert net.__dict__["_program_train"]._prepared == []
        with torch.no_grad():
            net(list(b))  # records the inference program
            net(list(b))
            assert net.prefetch(b[0])  # an inference entry
        net.train()
        net.load_state_dict(state)
        got, _ = _steps(net, [b], prefetch=False)
        _same(want, got)
        assert _count(TRAIN_PREPARED) == p0
        assert len(net.__dict__.get("_prefetched", ())) == 1
        torch.cuda.synchronize()
    finally:
        scn.set_math_mode("fp32")


def test_memory_flat_over_prefetched_steps():
    """20 steps with prefetch one step ahead, plus one prepared step per step that is never used (dropped when a third arrives):
    the library's memory pool and torch's allocations stop growing"""
    scn = _scn("bf16")
    try:
        net = _net(scn, "mini4")
        seq = [_inputs(bld) for bld in CASES["mini4"][1]]
        _record(net, seq[0])
        unused = [_inputs(bld)[0] for bld in CASES["mini4"][1]]
        chunks, mib, alloc = [], [], []
        assert net.prefetch(seq[0][0])
        for i in range(20):
            c, f = seq[i % 2]
            net.zero_grad(set_to_none=True)
            rpn, roi = net([c, f])
            assert net.prefetch(unused[i % 2])
            assert net.prefetch(seq[(i + 1) % 2][0])
            sum((m.features ** 2).mean() for m in rpn + roi).backward()
            del rpn, roi
            torch.cuda.synchronize()
            chunks.append(_count(CHUNKS))
            mib.append(_count(2))
            alloc.append(torch.cuda.memory_allocated())
        assert max(chunks[6:]) == chunks[6], chunks
        assert max(mib[6:]) == mib[6], mib
        assert max(alloc[6:]) == alloc[6], alloc
    finally:
        scn.set_math_mode("fp32")
