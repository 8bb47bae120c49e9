"""Developer tool: end-to-end error of each math mode against the reference's fp32 golden outputs."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fpn_util  # noqa: E402
import detection_3d_b200.sparseconvnet as scn  # noqa: E402
from detection_3d_b200 import synthetic  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
for name, cfg, bld in (("mini4", fpn_util.mini4_config(), dict(nx=60, ny=56, nz=24, n_walls=3, seed=3)),
                       ("sw4c_mid", scn.sw4c_fpn432_config(), dict(nx=300, ny=280, nz=40, n_walls=5, seed=5))):
    g = np.load(os.path.join(GOLD, f"fpn_{name}.npz"))
    for mode in ("fp32", "tf32", "tf32x3", "bf16"):
        scn.set_math_mode(mode)
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        net = net.cuda().eval()
        coords = synthetic.building_coords(**bld)
        feats = fpn_util.features_for(coords)
        with torch.no_grad():
            rpn, roi = net([torch.from_numpy(coords), torch.from_numpy(feats).cuda()])
        errs = []
        for tag, maps in (("rpn", rpn), ("roi", roi)):
            for i, m in enumerate(maps):
                ref = g[f"{tag}{i}_features"]
                got = m.features.cpu().numpy()
                errs.append((float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max())),
                             float(np.sqrt(((got - ref) ** 2).mean()) / max(1e-9, np.sqrt((ref ** 2).mean())))))
        print(name, mode, "max-abs/max:", ["%.2e" % e[0] for e in errs], "rel-rms:", ["%.2e" % e[1] for e in errs], flush=True)
scn.set_math_mode("fp32")
