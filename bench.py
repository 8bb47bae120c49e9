#!/usr/bin/env python
"""Benchmark of the Detection_3D sparse backbone path (BASELINE.json north_star).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--math tf32|bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one `FPN_Net.forward` of the sw_4c_fpn432 backbone (BASELINE.json configs[1]) on the
synthetic 470 m^2 building "B470" (1,177,224 input rows / 1,155,656 active voxels), INCLUDING the
Metadata / rulebook build, which the reference redoes every forward (sparseconvnet/ioLayers.py:52-55).
Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM.  `e2e`: same metric through the
public API with HOST (pinned) coords + features, H2D and D2H copies inside the timed region.
`--dump-outputs DIR`: the maps the last timed step returned, as DIR/<map>_features.npy (float32) and
DIR/<map>_locations.npy (float64: x, y, z, batch index per row); the inputs are seeded, so two builds
can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = ("sw_4c_fpn432 backbone forward incl. Metadata/rulebook build, one B470 synthetic building (1,155,656 active voxels) "
            "per GPU per step")  # the same string in both arms (the reference arm's per-step sample is stated in cpu_baseline.sample)
# end-to-end tolerance of each math mode against the reference's fp32 outputs (max |got - ref| / max(1, max|ref|) per returned
# map; the same numbers tests/test_gpu_pins.py states): exact fp32 / tf32 operands / bf16 operands
PARITY_TOL = {"fp32": 2e-4, "tf32": 1e-2, "bf16": 4.5e-2}  # measured on B470: 3.8e-6 / 4.0e-3 / 2.5-2.8e-2
B470_VOXELS = 1155656
B470_GMAC = 334.126  # SURVEY.md section 8(d): reference's own forward_pass_multiplyAdd_count for B470
# dominant kernel: m_mergeds.7 = SubmanifoldConvolution 128->128, 3^3, on level 0 (10,715,792 rules)
DOM_RULES, DOM_C = 10715792, 128


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        smax = next((float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()), None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """All host cores this process may use; exported as OMP_NUM_THREADS unconditionally (torchrun sets it to 1)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(n)
    return n


def cpu_reference_forward(coords, feats, cfg, state, keep=None):
    """One backbone forward on the host cores with the reference's own CPU code (oracle/_ref) when
    it was built, else with our C port of it.  Returns (seconds, macs, kind, threads); `keep`, a list,
    receives the returned maps (dicts: features, locations, spatial_size) for the parity check."""
    import torch
    from oracle import fpn_oracle, ref_python
    threads = host_threads()
    torch.set_num_threads(threads)  # (torchrun exports OMP_NUM_THREADS=1; host_threads() has already overridden it)
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "SCN.so"))
    fn = fpn_oracle.run_fpn_ref if have_ref else fpn_oracle.run_fpn_port
    t0 = time.perf_counter()
    rpn, roi, macs = fn(cfg, state, coords, feats)
    dt = time.perf_counter() - t0
    if keep is not None:
        keep[:] = rpn + roi
    return dt, macs, ("reference" if have_ref else "port"), threads


def config_of(n_gpus):
    """`config` of the JSON line -- the same object in both arms."""
    return {"workload": WORKLOAD, "l2": "256 MiB L2 flush between timed iterations (GPU arm)", "parallelism": f"replicas x{n_gpus}, no collective"}


def parity_of(maps, ref_maps, tol):
    """GPU step outputs (SparseConvNetTensors) against the reference's outputs of the same building (dicts from the
    cpu_baseline leg): identical row coordinates, and per returned map max |got - ref| / max(1, max|ref|) and relative rms."""
    import numpy as np
    worst, worst_rms, same_rows, per_map = 0.0, 0.0, True, []
    for m, r in zip(maps, ref_maps):
        got = m.features.float().cpu().numpy()
        ref = np.asarray(r["features"], dtype=np.float32)
        loc_ok = bool(np.array_equal(m.get_spatial_locations().numpy(), np.asarray(r["locations"])))
        same_rows = same_rows and loc_ok and got.shape == ref.shape
        if got.shape != ref.shape:
            per_map.append(None)
            continue
        err = float(np.abs(got - ref).max() / max(1.0, float(np.abs(ref).max()))) if ref.size else 0.0
        rms = float(np.sqrt(((got - ref).astype(np.float64) ** 2).mean()) / max(1e-30, np.sqrt((ref.astype(np.float64) ** 2).mean()))) if ref.size else 0.0
        worst, worst_rms = max(worst, err), max(worst_rms, rms)
        per_map.append(round(err, 6))
    return {"max_abs_over_max": worst, "rel_rms": worst_rms, "rows_identical": same_rows, "n_maps": len(ref_maps), "per_map": per_map,
            "tolerance": tol, "ok": bool(same_rows and len(maps) == len(ref_maps) and worst <= tol),
            "against": "reference CPU forward of the same full B470 building in this run (cpu_baseline leg)"}


def dump_outputs(out_dir, rpn, roi):
    """The maps FPN_Net.forward returned: features [rows, C] as float32, locations [rows, 4] as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for tag, maps in (("rpn", rpn), ("roi", roi)):
        for i, m in enumerate(maps):
            arrays[f"{tag}{i}_features"] = m.features.detach().float().cpu().numpy()
            arrays[f"{tag}{i}_locations"] = m.get_spatial_locations().numpy().astype(np.float64)
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "outputs exceed 64 MB"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_model(cfg, device):
    import torch
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    torch.manual_seed(0)
    net = scn.FPN_Net(**cfg)
    state = fpn_util.deterministic_state(net, seed=1)
    net.load_state_dict(state)
    return net.to(device).eval(), state


def run_reference_arm(args, rank, world):
    """--impl reference: the reference CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    host_threads()  # before torch / OpenMP start
    import numpy as np
    import fpn_util
    import detection_3d_b200.sparseconvnet.fpn as fpn
    from detection_3d_b200 import synthetic
    cfg = fpn.sw4c_fpn432_config()
    import torch
    net = fpn.FPN_Net(**cfg)
    state = fpn_util.deterministic_state(net, seed=1)
    # calibrate on a small crop, then size the per-step sample so the whole run stays within ~4 minutes
    cal = synthetic.building_coords(nx=136, ny=136, nz=68)
    tcal, _, kind, threads = cpu_reference_forward(cal, fpn_util.features_for(cal), cfg, state)
    ncal = np.unique(cal[:, :3], axis=0).shape[0]
    budget = 200.0 / max(1, args.steps + args.warmup)
    frac = min(1.0, max(0.02, budget / (tcal * B470_VOXELS / ncal)))
    nx = max(64, int(542 * frac ** 0.5))
    coords = synthetic.building_coords(nx=nx, ny=nx, nz=68) if frac < 1.0 else synthetic.building_coords()
    feats = fpn_util.features_for(coords)
    nvox = np.unique(coords[:, :3], axis=0).shape[0]
    times, macs = [], 0.0
    for i in range(args.warmup + args.steps):
        t, macs, kind, threads = cpu_reference_forward(coords, feats, cfg, state)
        if i >= args.warmup:
            times.append(t)
    step = sum(times) / len(times)
    value = (nvox / B470_VOXELS) / step  # B470-equivalent buildings per second
    sample = f"{nx}x{nx}x68 crop of B470 ({nvox} active voxels = {nvox / B470_VOXELS:.3f} building, {macs / 1e9:.1f} GMAC) per step; value scaled by voxel count"
    line = {
        "impl": "reference", "metric": "backbone_buildings_per_s", "value": value, "unit": "buildings/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_of(args.gpus),
        "cpu_baseline": {"value": value, "unit": "buildings/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "buildings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "tflops": 2 * macs / step / 1e12, "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def leg_batch64(args, rank, world, dev, net, n_build=64, steps=3):
    """BASELINE.json config 4: batched inference over 64 DISTINCT synthetic buildings (B470 footprint jittered +-15 %, seeds 0..63)
    sharded by building across the ranks (longest first, no collective on the data path).  Every rank streams its shard from
    pinned host memory through the backbone (Metadata built two buildings ahead) and copies every returned map back to pinned
    host memory.  Device-timed from a barrier to the last rank's completion; value = 64 / that time."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import fpn_util
    from detection_3d_b200 import distributed, synthetic
    dims = []
    for seed in range(n_build):
        rs = np.random.RandomState(1000 + seed)
        dims.append((int(542 * (1 + 0.15 * (2 * rs.rand() - 1))), int(542 * (1 + 0.15 * (2 * rs.rand() - 1)))))
    sizes = [2 * nx * ny + 16 * 68 * (nx + ny) // 2 for nx, ny in dims]
    mine = distributed.shard_buildings(sizes, world, rank)
    inputs = []
    for i in mine:
        c = synthetic.building_coords(nx=dims[i][0], ny=dims[i][1], nz=68, seed=i)
        inputs.append((i, torch.from_numpy(c).pin_memory(), torch.from_numpy(fpn_util.features_for(c)).pin_memory()))
    h2d = sum(c.numel() * 8 + f.numel() * 4 for _, c, f in inputs)
    depth = 2
    with torch.no_grad():
        warm = synthetic.building_coords(nx=624, ny=624, nz=68, seed=99)  # at least as large as any building of the batch
        wc, wf = torch.from_numpy(warm).pin_memory(), torch.from_numpy(fpn_util.features_for(warm)).pin_memory()
        net.reset_program()
        net([wc, wf])  # records the program
        for _ in range(2):
            net.prefetch(wc)
        for j in range(5):  # the Metadata / register pools reach their steady size
            rpn, roi = net([wc, wf])
            if j < 3:
                net.prefetch(wc)
        # pinned staging for every result of the shard, allocated up front (page-locking memory inside the loop costs milliseconds)
        per_building = sum(m.features.numel() for m in rpn + roi)
        stage = torch.empty(int(per_building * 1.3) * max(1, len(inputs)), dtype=torch.float32).pin_memory()
        pace = int(os.environ.get("BATCH_PACE", "1"))  # forwards the host may run ahead of the GPU (the Metadata builds run two buildings ahead regardless)

        def one_pass():
            stage_off, d2h, outs, done = 0, 0, {}, []
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for j in range(min(depth, len(inputs))):
                net.prefetch(inputs[j][1])
            for j, (i, c, f) in enumerate(inputs):
                if pace >= 0 and j - pace - 1 >= 0:
                    done[j - pace - 1].synchronize()
                rpn, roi = net([c, f])
                if j + depth < len(inputs):
                    net.prefetch(inputs[j + depth][1])
                got = []
                for m in rpn + roi:  # results go back to the host asynchronously
                    n_el = m.features.numel()
                    hbuf = (stage[stage_off:stage_off + n_el] if stage_off + n_el <= stage.numel() else torch.empty(n_el, dtype=torch.float32, pin_memory=True)).view(m.features.shape)
                    stage_off += n_el
                    hbuf.copy_(m.features, non_blocking=True)
                    d2h += n_el * 4
                    got.append(hbuf)
                outs[i] = got
                e = torch.cuda.Event()
                e.record()
                done.append(e)
            b.record()
            torch.cuda.synchronize()
            net.__dict__.pop("_prefetched", None)
            tp = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            return tp.item(), d2h, outs

        # the whole batch `steps` times (three by default): the first pass of a fresh process is occasionally 2-3x slower (cold host pages) and the host
        # side of this leg (5 GB of pinned uploads per pass) is sensitive to whatever else the box is doing; the best pass is reported,
        # all are listed
        passes = []
        for _ in range(steps):
            ms_p, d2h, outs = one_pass()
            passes.append(ms_p)
    t = torch.tensor([min(passes)], device=dev, dtype=torch.float64)
    ok = all(all(bool(torch.isfinite(h).all()) for h in v) for v in outs.values())
    counts = torch.tensor([len(inputs)], device=dev)
    if world > 1:
        dist.all_reduce(counts)
    ms = t.item()
    from detection_3d_b200._lib import lib
    pool = {"chunk_mallocs": lib().scn_debug_counter(0), "chunk_waits": lib().scn_debug_counter(1), "pool_mib": lib().scn_debug_counter(2)}
    return {"pool": pool, "ms_passes": passes, "steps": steps, "metric": "batched_inference_buildings_per_s", "value": n_build / (ms * 1e-3), "unit": "buildings/s", "buildings": n_build, "ms_total": ms,
            "ms_per_building": ms / n_build, "scaling": "strong", "buildings_done": int(counts.item()), "finite": ok,
            "h2d_bytes_rank0": h2d, "d2h_bytes_rank0": d2h, "shard_sizes": [len(distributed.shard_buildings(sizes, world, r)) for r in range(world)],
            "note": "64 distinct buildings (B470 +-15 %), host pinned inputs, sharded longest-first, Metadata built two buildings ahead, outputs copied to pinned host memory"}


def leg_rpn(args, rank, world, dev, net, coords_pin, feats_pin, steps=20, warmup=3):
    """BASELINE.json config 3: full sw_4c_fpn432 RPN inference per building -- backbone + FPN (the headline path), RPN head and anchors
    on the four rpn maps, then per class group sigmoid / top-1500 / box decode / rotated 3-D NMS / top-750 (tools/train_net_sparse3d.py:
    247-255) -- from pinned host inputs to the proposals on the host.  Random-init head (no checkpoint): the NMS work depends on the
    boxes, so the proposal counts are reported beside the time."""
    import torch
    import torch.distributed as dist
    from detection_3d_b200 import detector
    torch.manual_seed(0)
    det = detector.SparseRPNDetector(net, detector.RPNModule()).to(dev).eval()
    with torch.no_grad():
        # the default init (std 0.01) gives logits and box deltas of ~1e-3, i.e. all-equal scores and boxes = anchors: scale the layers so
        # that the outputs have the spread of a trained head (logits of a few units, deltas of ~0.2)
        det.rpn.head.conv.weight.mul_(10.0)
        det.rpn.head.cls_logits.weight.mul_(20.0)
        det.rpn.head.bbox_pred.weight.mul_(1.5)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        with torch.no_grad():
            groups = det([coords_pin, feats_pin])
            return [(b.bbox3d.to("cpu", non_blocking=True), b.get_field("objectness").to("cpu", non_blocking=True)) for gr in groups for b in gr]

    for _ in range(warmup):
        out = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.fill_(1)
        a.record()
        out = step()
        b.record()
    torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / steps
    n_anchor = sum(int(x) for x in [786, 1156, 289, 81]) * 4
    return {"metric": "rpn_inference_buildings_per_s", "value": world * 1e3 / ms, "unit": "buildings/s", "ms_per_step": ms, "steps": steps, "scaling": "weak",
            "anchors": n_anchor, "proposals_per_group": [int(o[0].shape[0]) for o in out], "finite": all(bool(torch.isfinite(o[0]).all()) for o in out),
            "note": "backbone + RPN head + anchors + per-group top-1500 / decode / rotated 3-D NMS (thresh 0.5) / top-750; pinned host inputs -> proposals on the host; "
                    "L2 flush between steps; random-init head"}


def leg_train(args, rank, world, dev, scn, steps=8, warmup=4):
    """BASELINE.json config 5: 6c_fpn4321 backbone training step (train-mode forward, loss = sum of squares of the returned maps,
    backward), batch 1 per GPU (one B470 building per rank, seed = rank), data-parallel gradient all-reduce over NCCL overlapped
    with the backward pass (distributed.GradientReducer).  CUDA-event times, max over ranks."""
    import torch
    import torch.distributed as dist
    import fpn_util
    from detection_3d_b200 import distributed, synthetic
    net = scn.FPN_Net(**scn.c6_fpn4321_config())
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net = net.to(dev).train()
    coords_np = synthetic.building_coords(seed=rank)
    coords = torch.from_numpy(coords_np).pin_memory()  # host coordinates as in the reference (ioLayers.py:60), page-locked: a pageable 37 MB copy blocks the host for ~3 ms
    feats = torch.from_numpy(fpn_util.features_for(coords_np)).to(dev)
    params = [p for p in net.parameters() if p.requires_grad]
    red = distributed.GradientReducer(params)
    times, loss, attached = [], None, False
    for it in range(warmup + steps):
        if not attached:  # from the second step on the backward pass writes into the reducer's buffer and signals per-parameter events
            attached = red.attach(net)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        if world > 1 and it == warmup:
            dist.barrier()
        ev[0].record()
        red.zero()
        rpn, roi = net([coords, feats])
        loss = sum((m.features ** 2).sum() for m in rpn + roi)
        ev[1].record()
        loss.backward()
        ev[2].record()
        n_coll = red.finish()
        ev[3].record()
        torch.cuda.synchronize()
        if it >= warmup:
            times.append([ev[i].elapsed_time(ev[i + 1]) for i in range(3)] + [ev[0].elapsed_time(ev[3])])
    t = torch.tensor(times, device=dev, dtype=torch.float64).mean(0)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # the collective alone: all-reduce of the whole flat gradient buffer, bus bandwidth = 2 (N-1)/N bytes / time
    bus = None
    if world > 1:
        for _ in range(2):
            dist.all_reduce(red.flat)
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            dist.all_reduce(red.flat)
        b.record()
        torch.cuda.synchronize()
        tt = torch.tensor([a.elapsed_time(b) / 5], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        bus = {"ms": tt.item(), "bytes": red.nbytes(), "bus_gbs": 2 * (world - 1) / world * red.nbytes() / (tt.item() * 1e-3) / 1e9}
    with_grad = sum(1 for p in params if p in (red.live or ()))
    out = {"metric": "train_steps_per_s", "value": world * 1e3 / t[3].item(), "unit": "buildings/s (fwd+bwd+allreduce, bs 1 per GPU)", "ms_per_step": t[3].item(),
           "forward_ms": t[0].item(), "backward_ms": t[1].item(), "allreduce_exposed_ms": t[2].item(), "collectives_per_step": n_coll,
           "gradient_bytes": red.nbytes(), "allreduce_alone": bus, "loss": float(loss), "params_with_grad": with_grad, "params": len(params),
           "scaling": "weak", "steps": steps, "math": {0: "fp32", 1: "tf32", 2: "bf16"}[scn.SCN.math_mode()],
           "replayed": bool(net.__dict__.get("_program_train") is not None), "program_backward_calls": int(scn.SCN.lib().scn_debug_counter(11)),
           "note": "6c_fpn4321 backbone, one B470 building per rank; first step layer by layer under autograd while the calls are recorded, later steps = ONE autograd node (scn_program_run in training mode + scn_program_backward) that writes the gradients straight into the reducer's flat buffer; every bucket's all-reduce waits for the events of its own parameters only (overlaps the rest of the backward pass)"}
    del net, red
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 400 for the headline = a >= 2 s steady-state window, 3 for the reference arm; --config rpn / train / batch64: 20 steps / 8 steps / 3 passes over the batch)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--math", default=os.environ.get("SCN_MATH", "auto"), choices=["auto", "fp32", "tf32", "bf16"])
    ap.add_argument("--config", default="backbone", choices=["backbone", "rpn", "batch64", "train"],
                    help="backbone = BASELINE.json configs[1] (the headline; its JSON line also carries batch64 / train sub-results unless --no-extras); "
                         "batch64 = config 4 alone; train = config 5 alone")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained leg and the tf32 / fp32 sub-results")
    ap.add_argument("--sustain-steps", type=int, default=400, help="steps of the steady-state leg (>= 2 s of back-to-back forwards)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the maps returned by the last timed step of the headline as DIR/<map>_{features,locations}.npy")
    args = ap.parse_args()
    steps_given = args.steps is not None  # configs rpn / batch64 / train keep their own step counts unless --steps is passed
    if args.steps is None:
        args.steps = 400 if args.impl == "ours" else 3
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "backbone"):
        ap.error("--dump-outputs writes the outputs of the headline (--impl ours --config backbone)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)
    # stdout carries exactly ONE line (the JSON): libraries that chat on fd 1 (NCCL prints its version there) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    import numpy as np
    import torch
    import torch.distributed as dist
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic

    if world > 1 and os.environ.get("BENCH_AFFINITY", "1") == "1" and hasattr(os, "sched_setaffinity"):
        # one process per GPU: give every rank its own slice of the host cores (main thread + the two build workers wake up on
        # GPU events dozens of times per forward; ranks migrating over each other's cores cost ~2 ms per step at N = 2)
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = len(cores) // world
            if per >= 4:  # main thread + three build workers; with fewer cores per rank the scheduler does better unpinned
                os.sched_setaffinity(0, cores[local * per:(local + 1) * per])
        except OSError:
            pass
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    math = args.math
    if math == "auto":  # bf16 operands / fp32 accumulate: the compute dtype the contract names; --math tf32 | fp32 for the others
        math = "bf16" if scn.SCN.lib().scn_tensor_core_path_available() else "fp32"
    scn.set_math_mode(math)

    cfg = scn.sw4c_fpn432_config()
    net, state = make_model(cfg, dev)
    if args.config != "backbone":  # configs 4 / 5 on their own: one JSON line in the same format
        leg_steps = {"steps": args.steps} if steps_given else {}
        if args.config == "rpn":
            c_np = synthetic.building_coords()
            sub = leg_rpn(args, rank, world, dev, net, torch.from_numpy(c_np).pin_memory(), torch.from_numpy(fpn_util.features_for(c_np)).pin_memory(), **leg_steps)
        else:
            sub = leg_batch64(args, rank, world, dev, net, **leg_steps) if args.config == "batch64" else leg_train(args, rank, world, dev, scn, **leg_steps)
        line = {"metric": sub.pop("metric"), "value": sub.pop("value"), "unit": sub.pop("unit"), "n_gpus": world, "steps": sub.get("steps", 1), "warmup": args.warmup,
                "ms_per_step": sub.get("ms_per_step", sub.get("ms_total")), "higher_is_better": True, "scaling": sub.pop("scaling"), "vs_baseline": None,
                "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[math], "data": "synthetic",
                "config": {"workload": {"batch64": "BASELINE.json config 4 (batch64)", "rpn": "BASELINE.json config 3 (backbone + FPN + RPN inference per building)",
                                        "train": "BASELINE.json config 5 (6c_fpn4321 training step)"}[args.config]},
                "detail": sub}
        if rank == 0:
            emit(line)
        if world > 1:
            dist.destroy_process_group()
        return
    coords_np = synthetic.building_coords()  # B470
    feats_np = fpn_util.features_for(coords_np)
    coords_dev = torch.from_numpy(coords_np).to(dev)
    feats_dev = torch.from_numpy(feats_np).to(dev)
    coords_pin = torch.from_numpy(coords_np).pin_memory()
    feats_pin = torch.from_numpy(feats_np).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_resident():
        with torch.no_grad():
            return net([coords_dev, feats_dev])

    def step_e2e():
        with torch.no_grad():
            # the reference's calling convention: coordinates stay a host LongTensor (ioLayers.py:60); the features are
            # handed over as a pinned host tensor too: the library copies the coordinates on its build stream and the
            # module queues the feature copy on the caller's stream right after
            rpn, roi = net([coords_pin, feats_pin])  # the module uploads both (coordinates first: the grid build needs them first)
            host = [m.features.to("cpu", non_blocking=True) for m in rpn + roi]
        return host

    def timed_stream(fn, coords_next, steps, warmup):
        """Streaming throughput: buildings are pushed through back to back; right after a forward has been queued the
        Metadata build of the NEXT building is started (FPN_Net.prefetch) so that it runs while the GPU computes the
        current one.  One event pair around all K steps, the L2 flushes included in the timed region."""
        net.__dict__.pop("_prefetched", None)
        fn()
        net.prefetch(coords_next)  # from here on the build runs two buildings ahead of the computation
        for _ in range(warmup):
            fn()
            net.prefetch(coords_next)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = scn.kernel_launch_count()
        a.record()
        for _ in range(steps):
            flush.fill_(1)  # L2 flush between iterations (inside the timed region)
            fn()
            net.prefetch(coords_next)
        b.record()
        torch.cuda.synchronize()
        launches = scn.kernel_launch_count() - l0
        if world > 1:
            dist.barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches

    def timed(fn, steps, warmup, keep=None):
        """`keep`, a list, receives what the last timed step returned."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = scn.kernel_launch_count()
        for i, (a, b) in enumerate(ev):
            flush.fill_(1)  # L2 flush between timed iterations (outside the event pair)
            a.record()
            if keep is not None and i == steps - 1:
                keep[:] = [fn()]
            else:
                fn()  # (outputs and their Metadata are released before the next step, as a caller's would be)
            b.record()
        torch.cuda.synchronize()
        launches = scn.kernel_launch_count() - l0
        if world > 1:
            dist.barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches

    sampler = ClockSampler(local)
    sampler.start()
    scn.forward_pass_multiplyAdd_count = 0
    last = []
    total_ms, launches = timed(step_resident, args.steps, args.warmup, keep=last)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # before any other forward can reuse the returned buffers
        dump_outputs(args.dump_outputs, *last[0])
    del last
    macs_per_step = scn.forward_pass_multiplyAdd_count / (args.steps + args.warmup)
    e2e_ms, _ = timed(step_e2e, args.steps, 1)
    # streaming variant (FPN_Net.prefetch builds the Metadata two buildings ahead); reported beside the headline, which
    # stays the plain one-building-at-a-time number
    stream_ms = None
    if world == 1:  # (single-process extra; the Metadata pool needs a few streamed steps to reach its steady size)
        stream_ms, _ = timed_stream(step_resident, coords_dev, args.steps, 6)
        net.__dict__.pop("_prefetched", None)
    ms_step = total_ms / args.steps
    value = world * 1e3 / ms_step
    # steady state: >= 2 s of back-to-back forwards with the clocks sampled over that window (a burst of 20 forwards at the
    # boost clock says little about a stream of buildings); when K itself is that long the headline IS the steady-state number
    sustained = None
    if not args.no_extras:
        if args.steps >= args.sustain_steps:
            sustained = {"steps": args.steps, "ms_per_step": ms_step, "value": value, "unit": "buildings/s", "seconds": total_ms / 1e3, "clocks": clocks,
                         "note": "the headline window itself"}
        else:
            smp = ClockSampler(local)
            smp.start()
            sus_ms, _ = timed(step_resident, args.sustain_steps, 0)
            sus_clocks = smp.stop()
            sustained = {"steps": args.sustain_steps, "ms_per_step": sus_ms / args.sustain_steps, "value": world * 1e3 / (sus_ms / args.sustain_steps),
                         "unit": "buildings/s", "seconds": sus_ms / 1e3, "clocks": sus_clocks,
                         "note": "same step as the headline, timed over a longer window right after it"}
    d2h = 0
    with torch.no_grad():
        rpn, roi = net([coords_dev, feats_dev])
        d2h = sum(m.features.numel() * 4 for m in rpn + roi)
        torch.cuda.synchronize()
    headline_maps = rpn + roi  # outputs of the very code path that was timed (replayed program, this math mode)

    # roofline of the dominant kernel, timed alone on the launching stream
    pk = peaks()
    roof = dominant_kernel_roofline(scn, torch, dev, coords_dev, flush, pk, math)

    line = {
        "metric": "backbone_buildings_per_s", "value": value, "unit": "buildings/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[math], "data": "synthetic",
        "numerics": {"fp32": "exact fp32 CUDA cores", "tf32": "tf32 operands, fp32 accumulate; end-to-end <= 1e-2 of max|ref| (tests)",
                     "bf16": "bf16 operands, fp32 accumulate, fp32 feature tensors at the API; end-to-end <= 4.5e-2 of max|ref| (tests + `parity` of this run)"}[math],
        "config": config_of(world), "sustained": sustained,
        "streaming": None if stream_ms is None else {
            "ms_per_step": stream_ms / args.steps, "value": world * 1e3 / (stream_ms / args.steps), "unit": "buildings/s",
            "note": "same forwards back to back with FPN_Net.prefetch building the Metadata two buildings ahead; L2 flush inside the timed region"},
        "tflops": value * 2 * macs_per_step / 1e12, "gmac_per_step": macs_per_step / 1e9,
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": world * 1e3 / (e2e_ms / args.steps), "unit": "buildings/s", "h2d_bytes_per_step": coords_np.nbytes + feats_np.nbytes, "d2h_bytes_per_step": d2h},
        "roofline": roof,
    }
    if not args.no_extras:  # BASELINE.json configs 4 and 5 ride along (same process group; a failing sub-leg never costs the headline)
        for name, fn in (("rpn", lambda: leg_rpn(args, rank, world, dev, net, coords_pin, feats_pin)), ("batch64", lambda: leg_batch64(args, rank, world, dev, net)),
                         ("train", lambda: leg_train(args, rank, world, dev, scn))):
            if name in os.environ.get("BENCH_SKIP", "").split(","):  # developer switch
                continue
            try:
                line[name] = fn()
            except Exception as e:
                line[name] = {"error": str(e)[:300]}
            net.reset_program()
            torch.cuda.empty_cache()
    parity_failed = False
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the reference's CPU forward of the SAME full building (6-7 s on 16 cores): the CPU baseline number, and its outputs are
        # what the GPU step's outputs are checked against, in every math mode measured
        ref_maps = []
        t, macs, kind, threads = cpu_reference_forward(coords_np, feats_np, cfg, state, keep=ref_maps)
        line["cpu_baseline"] = {"value": 1.0 / t, "unit": "buildings/s", "cores": threads, "kind": kind,
                                "sample": f"one forward of the full B470 building ({B470_VOXELS} voxels, {macs / 1e9:.1f} GMAC) in {t:.1f} s; outputs kept for `parity`"}
        line["parity"] = parity_of(headline_maps, ref_maps, PARITY_TOL[math])
        line["parity"]["macs_equal"] = bool(macs == macs_per_step)
        parity_failed = not line["parity"]["ok"]
        if not args.no_extras:  # the like-for-like precision modes, same building, same check
            modes = {}
            for other, k in (("tf32", 10), ("fp32", 3)):
                if other == math or (other != "fp32" and not scn.SCN.lib().scn_tensor_core_path_available()):
                    continue
                try:
                    scn.set_math_mode(other)
                    net.reset_program()
                    oms, _ = timed(step_resident, k, 3)
                    with torch.no_grad():
                        orpn, oroi = net([coords_dev, feats_dev])
                        torch.cuda.synchronize()
                    par = parity_of(orpn + oroi, ref_maps, PARITY_TOL[other])
                    modes[other] = {"ms_per_step": oms / k, "value": 1e3 / (oms / k), "unit": "buildings/s", "steps": k,
                                    "tflops": 1e3 / (oms / k) * 2 * macs_per_step / 1e12,
                                    "parity": {q: par[q] for q in ("max_abs_over_max", "rel_rms", "rows_identical", "tolerance", "ok")}}
                    parity_failed = parity_failed or not par["ok"]
                except Exception as e:  # a sub-result must never cost the headline
                    modes[other] = {"error": str(e)[:300]}
            scn.set_math_mode(math)
            net.reset_program()
            line["modes"] = modes
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    if parity_failed:
        sys.stderr.write("bench.py: PARITY FAILURE -- GPU outputs differ from the reference's beyond the stated tolerance: %s\n" % json.dumps(line.get("parity")))
        sys.exit(3)


def dominant_kernel_roofline(scn, torch, dev, coords_dev, flush, pk, math):
    """m_mergeds.7: SubmanifoldConvolution 128->128 3^3 on level 0 -- 175.6 of the 334.1 GMAC."""
    L = torch.LongTensor
    md = scn.Metadata(3)
    # rows numbered as in the timed forward: a replayed program runs on an internally numbered Metadata (row id = spatial rank,
    # DESIGN.md section 5), not in the reference's first-touch order of the (shuffled) input points
    from detection_3d_b200._lib import check, lib
    check(lib().scn_metadata_set_internal_numbering(md._h, 1))
    x0 = torch.empty(0, device=dev)
    scn.SCN.InputLayer_updateOutput(md, L([2048, 2048, 512]), coords_dev, torch.zeros(coords_dev.size(0), 1, device=dev), x0, 0, 4)
    n = md.getNActive(L([2048, 2048, 512]))
    x = torch.randn(n, DOM_C, device=dev)
    if math == "bf16":  # as inside the network: the producing BatchNorm / add kernel has already written the bf16 copy
        x._scn_bf16 = (x.to(torch.bfloat16), x._version)
    w = torch.randn(27, 1, DOM_C, DOM_C, device=dev) * 0.02
    out = torch.empty(0, device=dev)
    fwd = lambda: scn.SCN.SubmanifoldConvolution_updateOutput(L([2048, 2048, 512]), L([3, 3, 3]), md, x, out, w, torch.Tensor())
    macs = fwd()
    for _ in range(2):
        fwd()
    ts = []
    for _ in range(5):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fwd(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = sorted(ts)[len(ts) // 2]
    achieved = 2 * macs / (ms * 1e-3) / 1e12
    esz = 2 if math == "bf16" else 4
    # algorithmic HBM bytes of this launch (DESIGN.md 4.4): input rows once + output rows once + plan ids + weights
    alg_bytes = n * DOM_C * esz + n * DOM_C * 4 + 27 * n * 4 + 27 * DOM_C * DOM_C * esz
    # bytes the gathers pull through L2 (every rule fetches one input row) -- what actually bounds the kernel
    gather_bytes = DOM_RULES * DOM_C * esz
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_dominant_kernel_dram_bytes.json")
    if not os.path.exists(tp):
        tp = os.path.join(ROOT, "profiles", "r1_dominant_kernel_dram_bytes.json")
    if os.path.exists(tp):  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this launch
        traffic = json.load(open(tp)).get(math)
    return {"kernel": "conv_plan_tc (SubmanifoldConvolution 128->128 3^3, level 0: m_mergeds.7; rows in the internal numbering of the timed forward)", "bound": "tensor", "achieved": achieved,
            "peak": pk["tc_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tc_burst"], "peak_source": pk["src"] + " bf16 burst (kernel timed alone)",
            "ms_per_launch": ms, "algorithmic_flops": 2 * macs, "traffic": traffic, "algorithmic_hbm_bytes": alg_bytes,
            "hbm_gbs_if_compulsory_only": alg_bytes / (ms * 1e-3) / 1e9, "l2_gather_bytes": gather_bytes,
            "l2_gather_gbs": gather_bytes / (ms * 1e-3) / 1e9}


if __name__ == "__main__":
    main()
