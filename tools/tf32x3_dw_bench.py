"""What running the tf32x3 weight gradients on the tensor cores (split-operand conv_dw_tc, DESIGN.md section 4.6) gains over the
CUDA-core kernel k_dw, in one process:

  * share: the BASELINE.json config-5 training step (6c_fpn4321 on B470, replayed, no all-reduce) in tf32x3 under torch.profiler,
    one step in a run of its own: the summed kernel time of k_dw, of the split-operand path (k_split3_bf16 + conv_dw_tc) and of
    every kernel of the step;
  * layers: the weight gradient of single layers on B470 levels, one backward call each through the C ABI, k_dw (tf32 mode, where
    every weight gradient runs on it) against the split-operand path (tf32x3 mode), the two alternating, L2 overwritten before
    every call; the time is the summed duration of the weight-gradient kernels per call (torch.profiler), so the input gradients
    of the strided layers, which differ between the two modes, do not count; medians of the rounds;
  * step: the config-5 training step in tf32x3 and bf16, alternating, device events, medians of the rounds;
  * grads: the replayed 6c_fpn4321 training step on the 300 x 280 x 40 building (tests/test_gpu_tf32x3_dw.py) in tf32x3 against
    fp32 mode: max|d| / max|fp32 grad| of the worst parameters and the cosine of all gradients.  Run with --root on a checkout
    where tf32x3 weight gradients run on k_dw, it shows how much of the gap the weight-gradient kernel accounts for.

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON line.  --root runs the same
measurements against another checkout (a build of an earlier commit, where tf32x3 weight gradients all run on k_dw).

    python tools/tf32x3_dw_bench.py [--parts share,layers,step,grads] [--rounds 3] [--reps 5] [--train-steps 4] [--root DIR]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--parts", default="share,layers,step,grads")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--reps", type=int, default=5, help="profiled backward calls per layer, kernel and round")
ap.add_argument("--train-steps", type=int, default=4, help="timed training steps per mode and round")
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
args = ap.parse_args()
ROOT = os.path.abspath(args.root)
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True
DW_KERNELS = ("k_dw", "conv_dw_tc", "k_split3_bf16")
DW_RE = re.compile(r"\bscn::(k_dw|conv_dw_tc|k_split3_bf16)[<(]")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return [v.strip() for v in q.stdout.splitlines()[0].split(",")]
    except Exception as e:  # (the timing does not depend on it)
        return [f"unknown ({e})", "unknown", "unknown"]


def med(v):
    return sorted(v)[len(v) // 2]


def kernel_us(prof):
    """summed device time (us) per kernel name of a profiler session"""
    out = {}
    for e in prof.events():
        if str(e.device_type).endswith("CUDA"):
            out[e.name] = out.get(e.name, 0.0) + e.device_time
    return out


def dw_us(k):
    """the part of kernel_us that belongs to the weight-gradient kernels, per kernel"""
    out = dict.fromkeys(DW_KERNELS, 0.0)
    for name, v in k.items():
        m = DW_RE.search(name)
        if m:
            out[m.group(1)] += v
    return out


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic
    from detection_3d_b200._lib import check, l3, lib
    from gpu_adapter import GpuMetadata
    assert torch.cuda.is_available(), "needs a CUDA device"
    assert lib().scn_tensor_core_path_available(), "needs an sm_100 device"
    L = lib()
    dev = torch.device("cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    coords_np = synthetic.building_coords()  # B470
    coords = torch.from_numpy(coords_np).to(dev)
    feats = torch.from_numpy(fpn_util.features_for(coords_np)).to(dev)
    parts = args.parts.split(",")
    result = {"metric": "tf32x3_weight_gradient", "root": ROOT}

    tnets = {}

    def step(m):
        if m not in tnets:
            scn.set_math_mode(m)
            tnet = scn.FPN_Net(**scn.c6_fpn4321_config())
            tnet.load_state_dict(fpn_util.deterministic_state(tnet, seed=1))
            tnets[m] = tnet.to(dev).train()
        scn.set_math_mode(m)
        for p in tnets[m].parameters():
            p.grad = None
        rpn, roi = tnets[m]([coords, feats])
        sum((x.features ** 2).sum() for x in rpn + roi).backward()

    if "share" in parts:  # ---------------- kernel-time shares of one replayed tf32x3 step
        for _ in range(args.warmup):
            step("tf32x3")
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step("tf32x3")
            torch.cuda.synchronize()
        k = kernel_us(prof)
        total = sum(k.values())
        d = dw_us(k)
        result["share"] = {"kernel_ms_total": total / 1e3, "k_dw_ms": d["k_dw"] / 1e3, "k_dw_share": d["k_dw"] / total,
                           "split_operand_ms": (d["conv_dw_tc"] + d["k_split3_bf16"]) / 1e3,
                           "top": sorted(((n, v / 1e3) for n, v in k.items()), key=lambda t: -t[1])[:8]}
        scn.set_math_mode("fp32")

    if "layers" in parts:  # ---------------- single layers: k_dw (tf32 mode) against split operands (tf32x3)
        full = [2048, 2048, 512]
        G = GpuMetadata()
        G.input_layer(full, coords_np, 0, 4)
        sizes = [full]
        for _ in range(6):
            a = sizes[-1]
            b = [v // 2 for v in a]
            G.conv_rules(a, b, [2, 2, 2], [2, 2, 2])
            sizes.append(b)
        n = [int(G.nactive(s)) for s in sizes]
        h = G.m._h
        gen = torch.Generator(device=dev).manual_seed(0)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        layers = []

        def subm(lvl, cin, cout):
            x, dy, w = torch.randn(n[lvl], cin, device=dev, generator=gen), torch.randn(n[lvl], cout, device=dev, generator=gen), torch.zeros(27, cin, cout, device=dev)
            dw = torch.empty_like(w)
            return (f"subm {cin}->{cout} 3^3 level {lvl} ({n[lvl]} sites)",
                    lambda: check(L.scn_submanifold_convolution_backward(h, l3(sizes[lvl]), l3([3, 3, 3]), p(x), None, p(dy), p(w), p(dw), None, cin, cout)))

        for lvl in (0, 1, 2):
            layers += [subm(lvl, 128, 128), subm(lvl, 32, 32)]
        layers.append(subm(0, 9, 32))
        layers.append(subm(6, 128, 128))  # the deepest level: a few hundred rules per offset
        x, dy = torch.randn(n[0], 32, device=dev, generator=gen), torch.randn(n[1], 64, device=dev, generator=gen)
        w, dx = torch.zeros(8, 32, 64, device=dev), torch.empty(n[0], 32, device=dev)
        dws = torch.empty_like(w)
        layers.append((f"conv 32->64 2^3/2 level 0->1 ({n[0]} -> {n[1]} sites)",
                       lambda: check(L.scn_convolution_backward(h, l3(sizes[0]), l3(sizes[1]), l3([2, 2, 2]), l3([2, 2, 2]), p(x), p(dx), p(dy), p(w), p(dws), None, 32, 64))))
        xc, dyf = torch.randn(n[1], 64, device=dev, generator=gen), torch.randn(n[0], 32, device=dev, generator=gen)
        wd, dxc = torch.zeros(8, 64, 32, device=dev), torch.empty(n[1], 64, device=dev)
        dwd = torch.empty_like(wd)
        layers.append((f"deconv 64->32 2^3/2 level 1->0 ({n[1]} -> {n[0]} sites)",
                       lambda: check(L.scn_deconvolution_backward(h, l3(sizes[1]), l3(sizes[0]), l3([2, 2, 2]), l3([2, 2, 2]), p(xc), p(dxc), p(dyf), p(wd), p(dwd), None, 64, 32))))
        kern = {"k_dw": "tf32", "split_operand": "tf32x3"}
        res = {name: {kn: [] for kn in kern} for name, _ in layers}
        for name, f in layers:
            for m in kern.values():
                scn.set_math_mode(m)
                for _ in range(args.warmup):
                    f()
        torch.cuda.synchronize()
        for r in range(args.rounds):
            for name, f in layers:
                for kn, m in (list(kern.items()) if r % 2 == 0 else list(kern.items())[::-1]):
                    scn.set_math_mode(m)
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        for _ in range(args.reps):
                            flush.zero_()
                            f()
                        torch.cuda.synchronize()
                    d = dw_us(kernel_us(prof))
                    res[name][kn].append((d["k_dw"] if kn == "k_dw" else d["conv_dw_tc"] + d["k_split3_bf16"]) / args.reps / 1e3)
        scn.set_math_mode("fp32")
        result["layers_ms"] = {name: {kn: med(v) for kn, v in d.items()} for name, d in res.items()}
        result["layers_rounds_ms"] = res

    if "step" in parts:  # ---------------- config-5 training step, tf32x3 and bf16
        tmodes = ["tf32x3", "bf16"]
        tms = {m: [] for m in tmodes}
        for r in range(args.rounds):
            for m in tmodes:
                for _ in range(args.warmup if r == 0 else 1):
                    step(m)
                torch.cuda.synchronize()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.train_steps)]
                for a, b in ev:
                    a.record()
                    step(m)
                    b.record()
                torch.cuda.synchronize()
                tms[m].append(sum(a.elapsed_time(b) for a, b in ev) / args.train_steps)
        scn.set_math_mode("fp32")
        result["train_step_ms"] = {m: med(v) for m, v in tms.items()}
        result["train_step_rounds_ms"] = tms

    if "grads" in parts:  # ---------------- 6c_fpn4321 step gradients, tf32x3 against fp32 mode
        mc = synthetic.building_coords(nx=300, ny=280, nz=40, n_walls=5, seed=5)
        c, f = torch.from_numpy(mc), torch.from_numpy(fpn_util.features_for(mc)).to(dev)

        def grads(math):
            scn.set_math_mode(math)
            net = scn.FPN_Net(**scn.c6_fpn4321_config())
            state = fpn_util.deterministic_state(net, seed=1)
            net = net.to(dev).train()
            for _ in range(2):  # records, then replays
                net.load_state_dict(state)
                net.zero_grad(set_to_none=True)
                rpn, roi = net([c, f])
                sum((m.features ** 2).mean() for m in rpn + roi).backward()
            torch.cuda.synchronize()
            scn.set_math_mode("fp32")
            return {k: p.grad.double().cpu() for k, p in net.named_parameters() if p.grad is not None}

        want, got = grads("fp32"), grads("tf32x3")
        err = sorted(((float((got[k] - want[k]).abs().max() / max(1e-6, float(want[k].abs().max()))), k) for k in want), reverse=True)
        a, b = torch.cat([got[k].ravel() for k in sorted(want)]), torch.cat([want[k].ravel() for k in sorted(want)])
        result["grads_vs_fp32"] = {"worst": err[:4], "cosine": float(a @ b / (a.norm() * b.norm()))}

    name, power, clock = card()
    result.update({"gpu": name, "power_limit": power, "max_sm_clock": clock, "rounds": args.rounds, "reps": args.reps, "train_steps": args.train_steps})
    print(json.dumps(result))


if __name__ == "__main__":
    main()
