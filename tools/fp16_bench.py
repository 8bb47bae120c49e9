"""What the fp16 math mode (scn.set_math_mode("fp16"), DESIGN.md section 4.4) costs and how accurate it is, in one process:

  * the B470 headline forward (sw4c_fpn432, replayed program, inputs resident, L2 overwritten before each step as in bench.py) in
    bf16, fp16 and tf32 (fp32 for the error reference), the modes alternating round by round, medians over the rounds;
  * the dominant layer alone (submanifold 128 -> 128, 3x3x3, on level 0 of B470) in bf16 and fp16, same alternation;
  * the BASELINE.json config-5 training step (6c_fpn4321 on B470, replayed, no all-reduce) in bf16 and fp16;
  * max|d| / max|fp32| of every B470 output map of bf16, fp16 and tf32 against fp32 mode (worst map and every map);
  * range headroom: the largest |value| handed to a convolution (activations, weights) in the B470 forward, and to a convolution
    backward (rows and output gradients) in the config-5 training step at loss scale 1 -- everything the fp16 mode converts to
    fp16 is among these (an upper bound: layers that keep TF32 operands are included), to be read against fp16's 65504.

Prints one JSON line, with the card's name, power limit and maximum SM clock read in the same run.

    python tools/fp16_bench.py [--steps 20] [--layer-steps 50] [--train-steps 4] [--rounds 3]
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
    ap.add_argument("--steps", type=int, default=20, help="timed forwards per round and mode")
    ap.add_argument("--layer-steps", type=int, default=50, help="timed launches of the dominant layer per round and mode")
    ap.add_argument("--train-steps", type=int, default=4, help="timed training steps per round and mode")
    ap.add_argument("--rounds", type=int, default=3, help="rounds; the modes alternate inside each round")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    import fpn_util
    import detection_3d_b200.sparseconvnet as scn
    from detection_3d_b200 import synthetic
    from detection_3d_b200._lib import lib
    assert torch.cuda.is_available(), "needs a CUDA device"
    assert lib().scn_tensor_core_path_available(), "needs an sm_100 device"
    dev = torch.device("cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    coords_np = synthetic.building_coords()  # B470
    coords = torch.from_numpy(coords_np).to(dev)
    feats = torch.from_numpy(fpn_util.features_for(coords_np)).to(dev)
    result = {"metric": "fp16_cost_and_accuracy"}

    # ---------------- range headroom: layer-by-layer fp16 forward (B470) and training step (config 5) with the native calls watched
    from detection_3d_b200.sparseconvnet import native
    peak = {"forward": 0.0, "backward": 0.0}
    watch = {"forward": ["SubmanifoldConvolution_updateOutput", "Convolution_updateOutput", "Deconvolution_updateOutput",
                         "NetworkInNetwork_updateOutput"],
             "backward": ["SubmanifoldConvolution_backward", "Convolution_backward", "Deconvolution_backward",
                          "NetworkInNetwork_updateGradInput", "NetworkInNetwork_accGradParameters"]}
    orig = {}

    def watched(fn, phase):
        def f(*a, **k):
            for t in a:
                if isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.numel():
                    peak[phase] = max(peak[phase], float(t.abs().max()))
            return fn(*a, **k)
        return f
    for phase, names in watch.items():
        for nm in names:
            orig[nm] = getattr(native, nm)
            setattr(native, nm, watched(orig[nm], phase))
    try:
        scn.set_math_mode("fp16")
        net = scn.FPN_Net(**scn.sw4c_fpn432_config())
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        with torch.no_grad():
            net.to(dev).eval()([coords, feats])  # (the first forward runs layer by layer and records)
        fwd_peak = peak["forward"]
        tnet = scn.FPN_Net(**scn.c6_fpn4321_config())
        tnet.load_state_dict(fpn_util.deterministic_state(tnet, seed=1))
        rpn, roi = tnet.to(dev).train()([coords, feats])
        sum((x.features ** 2).sum() for x in rpn + roi).backward()
        torch.cuda.synchronize()
        result["fp16_range"] = {"b470_forward_max_abs": fwd_peak, "config5_backward_max_abs_loss_scale_1": peak["backward"], "fp16_max": 65504.0}
        del net, tnet, rpn, roi
    finally:
        for nm, fn in orig.items():
            setattr(native, nm, fn)
        scn.set_math_mode("fp32")
    torch.cuda.empty_cache()

    # ---------------- headline forward (one network per mode: each keeps its recorded program)
    modes = ["fp32", "bf16", "fp16", "tf32"]
    state = None
    nets = {}
    for m in modes:
        scn.set_math_mode(m)
        net = scn.FPN_Net(**scn.sw4c_fpn432_config())
        state = state or fpn_util.deterministic_state(net, seed=1)
        net.load_state_dict(state)
        nets[m] = net.to(dev).eval()

    def fwd(m):
        with torch.no_grad():
            rpn, roi = nets[m]([coords, feats])
        return [x.features for x in rpn + roi]

    ms = {m: [] for m in modes}
    outs = {}
    f16_launches = 0
    for r in range(args.rounds):
        for m in modes:
            scn.set_math_mode(m)
            for _ in range(args.warmup):
                out = fwd(m)
            torch.cuda.synchronize()
            c0 = lib().scn_debug_counter(18)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for a, b in ev:
                flush.fill_(1)
                a.record()
                out = fwd(m)
                b.record()
            torch.cuda.synchronize()
            if m == "fp16":
                f16_launches = (lib().scn_debug_counter(18) - c0) // args.steps
            outs[m] = [x.clone() for x in out]
            ms[m].append(sum(a.elapsed_time(b) for a, b in ev) / args.steps)
    per_map = {m: [float((x - y).abs().max() / max(1e-30, float(y.abs().max()))) for x, y in zip(outs[m], outs["fp32"])] for m in modes if m != "fp32"}
    err = {m: max(v) for m, v in per_map.items()}
    result["forward_ms"] = {m: med(ms[m]) for m in modes}
    result["forward_rounds_ms"] = ms
    result["forward_fp16_conv_launches"] = f16_launches
    result["b470_max_rel_err_vs_fp32"] = err
    result["b470_rel_err_vs_fp32_per_map"] = per_map
    del nets, out, outs
    torch.cuda.empty_cache()

    # ---------------- dominant layer alone: submanifold 128 -> 128, 3x3x3, level 0
    from gpu_adapter import GpuMetadata
    G = GpuMetadata()
    full = [2048, 2048, 512]
    n = G.input_layer(full, coords_np, 0, 4)
    rs = torch.Generator(device="cpu").manual_seed(0)
    x = torch.randn(n, 128, generator=rs).to(dev)
    w = (torch.randn(27, 1, 128, 128, generator=rs) * (2.0 / (128 * 27)) ** 0.5).to(dev)
    L = torch.LongTensor
    lms = {"bf16": [], "fp16": []}
    for r in range(args.rounds):
        for m in lms:
            scn.set_math_mode(m)
            o = torch.empty(0, device=dev)
            for _ in range(args.warmup):
                scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([3, 3, 3]), G.m, x, o, w, torch.Tensor())
            torch.cuda.synchronize()
            t = []
            for _ in range(args.layer_steps):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                scn.SCN.SubmanifoldConvolution_updateOutput(L(full), L([3, 3, 3]), G.m, x, o, w, torch.Tensor())
                b.record()
                t.append((a, b))
            torch.cuda.synchronize()
            lms[m].append(med([a.elapsed_time(b) for a, b in t]))
    result["layer0_128x128_rows"] = n
    result["layer0_128x128_ms"] = {m: med(v) for m, v in lms.items()}
    result["layer0_128x128_rounds_ms"] = lms
    del G, x, w, o
    torch.cuda.empty_cache()

    # ---------------- config-5 training step (single GPU, no all-reduce), bf16 and fp16
    tmodes = ["bf16", "fp16"]
    tnets = {}
    for m in tmodes:
        scn.set_math_mode(m)
        tnet = scn.FPN_Net(**scn.c6_fpn4321_config())
        tnet.load_state_dict(fpn_util.deterministic_state(tnet, seed=1))
        tnets[m] = tnet.to(dev).train()

    def step(m):
        params = [p for p in tnets[m].parameters() if p.requires_grad]
        for p in params:
            p.grad = None
        rpn, roi = tnets[m]([coords, feats])
        sum((x.features ** 2).sum() for x in rpn + roi).backward()

    tms = {m: [] for m in tmodes}
    for r in range(args.rounds):
        for m in tmodes:
            scn.set_math_mode(m)
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
    name, power, clock = card()
    result.update({"gpu": name, "power_limit": power, "max_sm_clock": clock,
                   "workloads": "B470 sw4c_fpn432 replayed forward (inputs resident, L2 overwritten before each step); submanifold 128 -> 128 3x3x3 "
                                "on B470 level 0 (L2 overwritten before each launch); B470 6c_fpn4321 replayed training step (no all-reduce)",
                   "steps": args.steps, "layer_steps": args.layer_steps, "train_steps": args.train_steps, "rounds": args.rounds})
    print(json.dumps(result))


if __name__ == "__main__":
    main()
