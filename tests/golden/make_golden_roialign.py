"""Generates tests/golden/roi_align_rotated_3d.npz for tests/test_gpu_pins.py::test_roi_align_rotated_3d_vs_restatement_and_golden.

A regression pin of the CPU restatement, not output of the reference's own kernels (those are compared live by
test_roi_align_rotated_3d_vs_reference_kernel where they have been built).  For every case of the test (same seeded inputs,
tests/test_gpu_pins.py::_roi_inputs) the densified, cropped map is built with the restatement (oracle/scn_oracle.c: InputLayer
mode 4 + SparseToDense) and ROIAlignRotated3D forward / backward are run on it with the restatement of the reference's kernels.

Stored per case and direction (`<case>_s<sampling>_fwd` / `_bwd`): the shape, max|.| of the whole array (the tolerance scale), and
the values at a fixed seeded sample of flat indices (`_idx`), half drawn from the non-zero entries and half from all entries.

  python tests/golden/make_golden_roialign.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import scn_oracle as so  # noqa: E402
from test_gpu_pins import _roi_inputs  # noqa: E402

N_SAMPLE = 4096  # per half: keeps the file well under 1 MB


def sample(a, rs):
    flat = a.ravel()
    nz = np.flatnonzero(flat)
    idx = np.concatenate([rs.choice(nz, min(N_SAMPLE, nz.size), replace=False), rs.choice(flat.size, min(N_SAMPLE, flat.size), replace=False)])
    return np.unique(idx).astype(np.int32)


def main():
    out = {}
    rs = np.random.RandomState(0)
    for case in ("small2", "level4"):
        for sampling in (2, 0):
            coords, feats, sz, C_, pooled, scale, ext, batch, rois, g = _roi_inputs(case, sampling)
            O = so.OracleMetadata()
            O.input_layer(sz, coords, 0, 4)
            hdr, tab = O.input_rules()
            rows = so.o_input_layer_forward(feats, hdr, tab)
            dense = so.o_sparse_to_dense_forward(rows, O.sparse_to_dense_rules(sz), sz)[:, :, :ext[0], :ext[1], :ext[2]]
            assert dense.shape == (batch, C_) + tuple(ext)
            fwd = so.o_roi_align_rotated_3d_forward(dense, rois, scale, pooled, sampling)
            bwd = so.o_roi_align_rotated_3d_backward(g, rois, scale, pooled, sampling, dense.shape)
            for key, a in ((f"{case}_s{sampling}_fwd", fwd), (f"{case}_s{sampling}_bwd", bwd)):
                idx = sample(a, rs)
                out[key + "_shape"] = np.array(a.shape, np.int64)
                out[key + "_absmax"] = np.float32(np.abs(a).max())
                out[key + "_idx"] = idx
                out[key] = a.ravel()[idx]
    np.savez_compressed(os.path.join(HERE, "roi_align_rotated_3d.npz"), **out)
    print({k: v.shape for k, v in out.items() if k.endswith("_idx")})


if __name__ == "__main__":
    main()
