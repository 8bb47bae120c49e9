"""The caller's Metadata after a replayed forward.

A replayed inference forward computes on an internally numbered Metadata and numbers the caller's Metadata beside it as an
overlay over the internal grids (reference row ids only; rulebooks built on first use).  Afterwards the caller's Metadata
must still be exactly the reference's: every rulebook, iteration order and location digest equals the digests taken from
the reference's own Metadata<3> (tests/golden/rulebooks.json), including the strided rulebooks whose output grid the
overlay created."""
import json
import os

import pytest
import torch

import fpn_util
from gpu_adapter import GpuMetadata
from detection_3d_b200 import synthetic

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
COORD_UPLOADS = 17  # scn_debug_counter: host -> device copies of input-layer coordinates

BUILDINGS = [
    ("mini4", dict(nx=60, ny=56, nz=24, n_walls=3, seed=3), [64, 64, 32], 4, (1, 2)),
    ("sw4c_mid", dict(nx=300, ny=280, nz=40, n_walls=5, seed=5), [2048, 2048, 512], 9, (4, 5, 6)),
    ("b470", dict(), [2048, 2048, 512], 9, (4, 5, 6)),
]


class ReturnedMetadata(GpuMetadata):
    """The adapter over a Metadata that came back with a forward's outputs."""

    def __init__(self, m):
        self.m = m


def _net(name):
    import detection_3d_b200.sparseconvnet as scn
    cfg = fpn_util.mini4_config() if name == "mini4" else scn.sw4c_fpn432_config()
    net = scn.FPN_Net(**cfg)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    return net.cuda().eval()


def _replayed_metadata(net, coords, feats):
    """Metadata returned with the outputs of a replayed forward (the first forward of a network records the program)."""
    with torch.no_grad():
        if net.__dict__.get("_program") is None:
            net([coords, feats])  # records
            assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
        rpn, roi = net([coords, feats])  # replays
    torch.cuda.synchronize()
    md = rpn[0].metadata
    assert all(m.metadata is md for m in rpn + roi)
    return md


def _check_against_golden(name, md, full, nl, pro, n_rows):
    gold = json.load(open(os.path.join(GOLD, "rulebooks.json")))[name]
    G = ReturnedMetadata(md)
    got = fpn_util.metadata_digests(G, full, nl, pro)
    got["input_rules"] = fpn_util.rulebook_digest(G.input_rules())
    got["n_input_rows"] = n_rows
    bad = {k: (got.get(k), gold[k]) for k in gold if got.get(k) != gold[k]}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("name,bld,full,nl,pro", BUILDINGS)
def test_metadata_after_replay_vs_reference_golden(name, bld, full, nl, pro):
    coords = synthetic.building_coords(**bld)
    c = torch.from_numpy(coords).cuda()
    f = torch.from_numpy(fpn_util.features_for(coords)).cuda()
    md = _replayed_metadata(_net(name), c, f)
    _check_against_golden(name, md, full, nl, pro, int(coords.shape[0]))


@pytest.mark.gpu
def test_metadata_after_replay_with_host_coordinates():
    """Host coordinates (the reference's calling convention): the internally numbered Metadata uploads them once; the
    overlay takes everything from it and uploads nothing."""
    import detection_3d_b200.sparseconvnet as scn
    name, bld, full, nl, pro = BUILDINGS[1]
    coords = synthetic.building_coords(**bld)
    c = torch.from_numpy(coords)
    f = torch.from_numpy(fpn_util.features_for(coords)).cuda()
    net = _net(name)
    with torch.no_grad():
        net([c, f])  # records
    assert net.__dict__.get("_program") is not None, net.__dict__.get("_program_error")
    torch.cuda.synchronize()
    before = scn.SCN.lib().scn_debug_counter(COORD_UPLOADS)
    md = _replayed_metadata(net, c, f)
    assert scn.SCN.lib().scn_debug_counter(COORD_UPLOADS) - before == 1
    _check_against_golden(name, md, full, nl, pro, int(coords.shape[0]))
