"""What a filter of more than 64 offsets costs (DESIGN.md section 8): a 64 -> 64 submanifold convolution with a 5x5x5 filter
(K = 125: two chunked conv_plan_tc launches, section 4.4) on level 0 of the B470 building, against the 3x3x3 layer of the same width,
in each math mode.  The two filters and the modes alternate inside each round; medians over the rounds.  Reports per layer and
mode the time, the rules per second (rules = (input row, output row) pairs of the rulebook, i.e. multiply-adds / (64 x 64)) and the
5^3 rate relative to the 3^3 rate.  Input rows are resident; the L2 (126 MB) is overwritten before every timed launch.

Prints one JSON line, with the card's name, power limit and maximum SM clock read in the same run.

    python tools/large_filter_bench.py [--steps 20] [--rounds 3] [--warmup 3]
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return [v.strip() for v in q.stdout.splitlines()[0].split(",")]
    except Exception as e:  # (the timing does not depend on it)
        return [f"unknown ({e})", "unknown", "unknown"]


def med(v):
    return sorted(v)[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed launches per round, filter and mode")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import ctypes as C
    import torch
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic
    from detection_3d_b200._lib import lib, check, l3
    from gpu_adapter import GpuMetadata
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda")
    modes = ["fp32", "tf32", "tf32x3", "bf16"] if lib().scn_tensor_core_path_available() else ["fp32"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    coords_np = synthetic.building_coords()  # B470
    full = [2048, 2048, 512]
    G = GpuMetadata()
    n = G.input_layer(full, coords_np, 0, 4)
    gen = torch.Generator(device="cpu").manual_seed(0)
    x = torch.randn(n, 64, generator=gen).to(dev)
    filters = {"3x3x3": 3, "5x5x5": 5}
    weights = {k: (torch.randn(f ** 3, 1, 64, 64, generator=gen) * (2.0 / (64 * f ** 3)) ** 0.5).to(dev) for k, f in filters.items()}
    rules = {}
    for k, f in filters.items():
        r = C.c_long()
        check(lib().scn_submanifold_prepare(G.m._h, l3(full), l3([f] * 3), C.byref(r)))
        rules[k] = r.value
    L = torch.LongTensor
    ms = {(k, m): [] for k in filters for m in modes}
    chunked = {}
    for _ in range(args.rounds):
        for m in modes:
            scn.set_math_mode(m)
            for k, f in filters.items():
                o = torch.empty(0, device=dev)
                for _ in range(args.warmup):
                    scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([f] * 3), G.m, x, o, weights[k], torch.Tensor())
                torch.cuda.synchronize()
                c0 = lib().scn_debug_counter(16)
                t = 0.0
                for _ in range(args.steps):
                    flush.fill_(1)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([f] * 3), G.m, x, o, weights[k], torch.Tensor())
                    b.record()
                    torch.cuda.synchronize()
                    t += a.elapsed_time(b)
                chunked[(k, m)] = (lib().scn_debug_counter(16) - c0) // args.steps
                ms[(k, m)].append(t / args.steps)
    scn.set_math_mode("fp32")
    name, power, clock = card()
    res = {"metric": "large_filter_cost", "gpu": name, "power_limit": power, "max_sm_clock": clock, "sites": n, "channels": 64,
           "rules": rules, "layers": {}}
    for m in modes:
        row = {}
        for k in filters:
            t = med(ms[(k, m)])
            row[k] = {"ms": round(t, 4), "rules_per_s": rules[k] / (t * 1e-3), "chunked_launches": chunked[(k, m)], "rounds_ms": ms[(k, m)]}
        row["5x5x5_rate_vs_3x3x3"] = row["5x5x5"]["rules_per_s"] / row["3x3x3"]["rules_per_s"]
        res["layers"][m] = row
    print(json.dumps(res))


if __name__ == "__main__":
    main()
