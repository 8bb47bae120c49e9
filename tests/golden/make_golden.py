"""Generates tests/golden/*.npz / *.json from the REFERENCE ITSELF (build container only).

  python tests/golden/make_golden.py

 * fpn_<name>.npz      outputs of the reference's own scn.FPN_Net (real Python package from
                       /root/reference on top of oracle/_ref/SCN.so) for a deterministic state_dict
                       and a seeded synthetic building: features + spatial locations of every
                       returned map, and the multiply-add counter.
 * fpn_mini4_train.npz one training step of the reference's scn.FPN_Net (train-mode forward, loss, autograd backward):
                       parameter gradients and BatchNorm buffers.  At 1.8 MB it is a known exception to the 1 MB kept
                       for test vectors: the training-step test bounds the worst element and the rms of every
                       gradient tensor and the cosine of the whole gradient vector, so it is stored whole, not sampled.
 * sparse_to_dense.npz scn.SparseToDense forward / backward and sparse_3d_to_dense_2d of the reference on a two-item batch.
 * rulebooks.json      sha1 digests of every grid / iteration order / rulebook of the reference's
                       own Metadata<3> (oracle/_ref/libscn_ref_rules.so) for three buildings,
                       including the full-size B470 building of BASELINE.json.
 * rulebook_small.npz  full rulebook arrays for a tiny case (readable by eye) + hash KATs.
Inputs are not stored: they are regenerated from the same seeded generators.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import fpn_util  # noqa: E402
from detection_3d_b200 import synthetic  # noqa: E402
from detection_3d_b200.sparseconvnet.fpn import sw4c_fpn432_config  # noqa: E402
from oracle import ref_python, scn_oracle  # noqa: E402

CASES = {
    "mini4": (fpn_util.mini4_config(), dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)),
    "sw4c_mid": (sw4c_fpn432_config(), dict(nx=300, ny=280, nz=40, n_walls=5, seed=5)),
}


def run_reference_fpn(name):
    cfg, bld = CASES[name]
    scn = ref_python.load_reference_package()
    args, kw = fpn_util.ref_ctor_args(cfg)
    net = scn.FPN_Net(*args, **kw)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net.eval()
    coords = synthetic.building_coords(**bld)
    feats = fpn_util.features_for(coords)
    scn.forward_pass_multiplyAdd_count = 0
    with torch.no_grad():
        rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats)])
    out = {"macs": np.float64(scn.forward_pass_multiplyAdd_count), "n_rpn": len(rpn), "n_roi": len(roi)}
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        for i, m in enumerate(maps):
            out[f"{tag}{i}_features"] = m.features.numpy().astype(np.float32)
            out[f"{tag}{i}_locations"] = m.get_spatial_locations().numpy().astype(np.int32)
            out[f"{tag}{i}_spatial_size"] = m.spatial_size.numpy().astype(np.int64)
    np.savez_compressed(os.path.join(HERE, f"fpn_{name}.npz"), **out)
    print(name, "macs", float(out["macs"]), {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim == 2})


def run_reference_fpn_train(name="mini4"):
    """Whole-network TRAINING step of the reference's own scn.FPN_Net through its autograd Functions (CPU extension):
    train-mode forward (batch statistics, running statistics updated), loss = sum over the returned maps of mean(f^2),
    backward.  Stored: the loss, every parameter gradient (None for the dead top-down levels, recorded as absent) and
    the BatchNorm buffers after the step."""
    cfg, bld = CASES[name]
    cfg = dict(cfg, track_running_stats=True)
    scn = ref_python.load_reference_package()
    args, kw = fpn_util.ref_ctor_args(cfg)
    net = scn.FPN_Net(*args, **kw)
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net.train()
    coords = synthetic.building_coords(**bld)
    feats = fpn_util.features_for(coords)
    rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats)])
    maps = rpn + roi
    loss = sum((m.features ** 2).mean() for m in maps)
    loss.backward()
    out = {"loss": np.float64(loss.item()), "n_maps": len(maps)}
    out["map_mean_sq"] = np.array([float((m.features ** 2).mean()) for m in maps], np.float64)  # (the loss terms; eval-mode features are in fpn_<name>.npz)
    n_grad = 0
    for k, p_ in net.named_parameters():
        if p_.grad is not None:
            out["grad:" + k] = p_.grad.numpy().astype(np.float32)
            n_grad += 1
    for k, b in net.named_buffers():
        out["buf:" + k] = b.numpy().astype(np.float32)
    np.savez_compressed(os.path.join(HERE, f"fpn_{name}_train.npz"), **out)
    print(name, "train: loss", float(out["loss"]), "params with grad", n_grad, "of", len(list(net.parameters())))


def run_reference_sparse_to_dense():
    """scn.SparseToDense forward + backward and tools_3d_2d.sparse_3d_to_dense_2d of the reference package on a two-item batch."""
    scn = ref_python.load_reference_package()
    rs = np.random.RandomState(21)
    coords = np.concatenate([np.concatenate([rs.randint(0, [12, 14, 6], (300, 3)), np.zeros((300, 1), np.int64)], 1),
                             np.concatenate([rs.randint(0, [9, 16, 8], (200, 3)), np.ones((200, 1), np.int64)], 1)]).astype(np.int64)
    feats = rs.randn(coords.shape[0], 6).astype(np.float32)
    inp = scn.InputLayer(3, torch.LongTensor([16, 16, 8]), mode=4)
    f = torch.from_numpy(feats).requires_grad_(True)
    x = inp([torch.from_numpy(coords), f])
    dense = scn.SparseToDense(3, 6)(x)
    w = torch.from_numpy(rs.randn(*dense.shape).astype(np.float32))
    (dense * w).sum().backward()
    sys.modules.setdefault("sparseconvnet", scn)
    from sparseconvnet.tools_3d_2d import sparse_3d_to_dense_2d
    crop = sparse_3d_to_dense_2d(x)
    np.savez_compressed(os.path.join(HERE, "sparse_to_dense.npz"), coords=coords, feats=feats, dense=dense.detach().numpy(), w=w.numpy(),
                        grad_feats=f.grad.numpy(), crop=crop.detach().numpy(), locations=x.get_spatial_locations().numpy(),
                        rows=x.features.detach().numpy())
    print("sparse_to_dense", tuple(dense.shape), tuple(crop.shape))


def rulebook_digests():
    res = {}
    cases = {
        "mini4": (dict(nx=60, ny=56, nz=24, n_walls=3, seed=3), [64, 64, 32], 4, (1, 2)),
        "sw4c_mid": (dict(nx=300, ny=280, nz=40, n_walls=5, seed=5), [2048, 2048, 512], 9, (4, 5, 6)),
        "b470": (dict(), [2048, 2048, 512], 9, (4, 5, 6)),
    }
    for name, (bld, full, nl, pro) in cases.items():
        coords = synthetic.building_coords(**bld)
        md = scn_oracle.RefMetadata()
        n = md.input_layer(full, coords, 0, 4)
        d = fpn_util.metadata_digests(md, full, nl, pro)
        d["input_rules"] = fpn_util.rulebook_digest(md.input_rules())
        d["n_input_rows"] = int(coords.shape[0])
        res[name] = d
        print(name, n, [d[f"n{l}"] for l in range(nl)])
    with open(os.path.join(HERE, "rulebooks.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)


def small_rulebook():
    # the 7-row example of SURVEY.md A.7 plus a batch-of-2 case
    coords = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [3, 3, 3], [2, 3, 3], [1, 0, 0]], np.int64)
    md = scn_oracle.RefMetadata()
    md.input_layer([8, 8, 8], coords, 0, 4)
    out = {"coords": coords}
    for i, a in enumerate(md.input_rules()):
        out[f"input{i}"] = a
    out["iter"] = md.iteration_order([8, 8, 8], 0)
    for k, a in enumerate(md.submanifold_rules([8, 8, 8], [3, 3, 3])):
        out[f"subm{k}"] = a
    for k, a in enumerate(md.conv_rules([8, 8, 8], [4, 4, 4], [2, 2, 2], [2, 2, 2])):
        out[f"conv{k}"] = a
    out["loc4"] = md.spatial_locations([4, 4, 4])
    for k, a in enumerate(md.conv_rules([4, 4, 4], [4, 4, 1], [1, 1, 4], [1, 1, 1])):
        out[f"pro{k}"] = a
    pts = np.array([[0, 0, 0], [1, 2, 3], [100, 200, 30], [541, 541, 67], [4095, 4095, 511], [-1, 0, 0]], np.int64)
    out["hash_points"] = pts
    out["hash_values"] = np.array([scn_oracle.rlib().ref_point_hash(int(a), int(b), int(c)) & 0xffffffff for a, b, c in pts], np.uint64)
    np.savez_compressed(os.path.join(HERE, "rulebook_small.npz"), **out)


if __name__ == "__main__":
    assert ref_python.available() and scn_oracle.have_ref(), "run `make -C oracle ref` first (needs /root/reference)"
    small_rulebook()
    rulebook_digests()
    for name in CASES:
        run_reference_fpn(name)
    run_reference_fpn_train("mini4")
    run_reference_sparse_to_dense()
