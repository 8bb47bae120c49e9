"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True), DESIGN.md section 7) on the two benchmarked workloads, in
one process: the B470 headline forward (sw4c_fpn432, bf16, replayed program, inputs resident, L2 overwritten between steps as in
bench.py) and the BASELINE.json config-5 training step (6c_fpn4321 on B470, bf16, replayed, no all-reduce), each timed with the flag
off and on in alternating rounds.  Every output of the timed deterministic steps is compared bitwise with the first one; the
largest difference between the two modes is reported as max|d| / max|x| per map (forward) or per gradient (training).  Prints one
JSON line, with the card name and power limit read in the same run.

    python tools/deterministic_bench.py [--steps 20] [--train-steps 4] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [v.strip() for v in q.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # (the timing does not depend on it)
        return f"unknown ({e})", "unknown"


def rel_diff(a, b):
    return float((a - b).abs().max() / max(1e-30, float(b.abs().max())))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed forwards per round and mode")
    ap.add_argument("--train-steps", type=int, default=4, help="timed training steps per round and mode")
    ap.add_argument("--rounds", type=int, default=3, help="off / on rounds (alternating)")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda")
    scn.set_math_mode("bf16")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    coords_np = synthetic.building_coords()  # B470
    coords = torch.from_numpy(coords_np).to(dev)
    feats = torch.from_numpy(fpn_util.features_for(coords_np)).to(dev)

    # ---------------- headline forward
    net = scn.FPN_Net(**scn.sw4c_fpn432_config())
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net = net.to(dev).eval()

    def fwd():
        with torch.no_grad():
            rpn, roi = net([coords, feats])
        return [m.features for m in rpn + roi]

    ms = {False: [], True: []}
    ref = {False: None, True: None}
    repeat_ok = True
    for r in range(args.rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            for _ in range(args.warmup):
                out = fwd()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for a, b in ev:
                flush.fill_(1)
                a.record()
                out = fwd()
                b.record()
                if det:  # every deterministic output against the first one (the comparison runs outside the event pair)
                    if ref[True] is None:
                        ref[True] = [x.clone() for x in out]
                    repeat_ok &= all(torch.equal(x, y) for x, y in zip(out, ref[True]))
            torch.cuda.synchronize()
            if ref[det] is None:
                ref[det] = [x.clone() for x in out]
            ms[det].append(sum(a.elapsed_time(b) for a, b in ev) / args.steps)
    fwd_diff = max(rel_diff(x, y) for x, y in zip(ref[True], ref[False]))
    del net, out, ref
    torch.cuda.empty_cache()

    # ---------------- config-5 training step (single GPU, no all-reduce)
    tnet = scn.FPN_Net(**scn.c6_fpn4321_config())
    tnet.load_state_dict(fpn_util.deterministic_state(tnet, seed=1))
    tnet = tnet.to(dev).train()
    params = [p for p in tnet.parameters() if p.requires_grad]

    def step():
        for p in params:
            p.grad = None
        rpn, roi = tnet([coords, feats])
        sum((m.features ** 2).sum() for m in rpn + roi).backward()
        return [p.grad for p in params if p.grad is not None]

    tms = {False: [], True: []}
    tref = {False: None, True: None}
    train_repeat_ok = True
    for r in range(args.rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            for _ in range(args.warmup if r == 0 else 1):
                grads = step()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.train_steps)]
            for a, b in ev:
                a.record()
                grads = step()
                b.record()
                if det:
                    if tref[True] is None:
                        tref[True] = [g.clone() for g in grads]
                    train_repeat_ok &= all(torch.equal(x, y) for x, y in zip(grads, tref[True]))
            torch.cuda.synchronize()
            if tref[det] is None:
                tref[det] = [g.clone() for g in grads]
            tms[det].append(sum(a.elapsed_time(b) for a, b in ev) / args.train_steps)
    train_diff = max(rel_diff(x, y) for x, y in zip(tref[True], tref[False]))
    torch.use_deterministic_algorithms(False)
    name, power = card()
    med = lambda v: sorted(v)[len(v) // 2]
    print(json.dumps({
        "metric": "deterministic_mode_cost", "gpu": name, "power_limit": power, "math": "bf16",
        "forward_ms": {"off": med(ms[False]), "on": med(ms[True]), "rounds_off": ms[False], "rounds_on": ms[True]},
        "forward_overhead": med(ms[True]) / med(ms[False]) - 1,
        "forward_on_bitwise_repeatable": bool(repeat_ok), "forward_max_rel_diff_on_vs_off": fwd_diff,
        "train_step_ms": {"off": med(tms[False]), "on": med(tms[True]), "rounds_off": tms[False], "rounds_on": tms[True]},
        "train_overhead": med(tms[True]) / med(tms[False]) - 1,
        "train_on_bitwise_repeatable": bool(train_repeat_ok), "train_max_rel_diff_on_vs_off": train_diff,
        "workloads": "B470 sw4c_fpn432 replayed forward (inputs resident, L2 overwritten before each step); B470 6c_fpn4321 replayed training step (no all-reduce)",
        "steps": args.steps, "train_steps": args.train_steps, "rounds": args.rounds}))


if __name__ == "__main__":
    main()
