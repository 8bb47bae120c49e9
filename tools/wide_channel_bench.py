"""What the tensor-core paths for layers wider than 256 channels (column slabs, channel-blocked weight gradients; DESIGN.md section
4.4) gain over the CUDA-core kernel those layers ran on before, in one process:

  * representative wide layers on B470 levels, one forward call each through the C ABI: 512 -> 512 3^3 submanifold on levels 4-6,
    256 -> 512 2^3 / 2 strided convolution (level 3 -> 4), 288 -> 288 2^3 / 2 deconvolution with a 288-channel lateral 1x1x1 stage
    (levels 1-3).  Modes bf16, fp16, tf32, tf32x3 against fp32 (for these shapes the fp32 mode runs the CUDA-core kernel every mode
    ran before), alternating within each round, L2 overwritten before every timed call, device events, medians of the rounds;
    TFLOP/s from the rule counts (2 x rules x Cin x Cout) and the share of the dense BF16 data-sheet peak (2,250 TFLOP/s, one B200);
  * the headline network widened (sw4c_fpn432 with nPlanesF = [32, 64, 64, 128, 320, 320, 512, 512, 512], nPlaneM = 288) on B470:
    the replayed forward and the replayed training step per mode.

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON line.

    python tools/wide_channel_bench.py [--rounds 3] [--reps 10] [--steps 6] [--train-steps 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True
MODES = {"fp32": 0, "tf32": 1, "bf16": 2, "tf32x3": 3, "fp16": 5}
BF16_PEAK = 2250e12


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
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10, help="timed calls per layer, mode and round")
    ap.add_argument("--steps", type=int, default=6, help="timed replayed forwards per mode and round")
    ap.add_argument("--train-steps", type=int, default=3, help="timed replayed training steps per mode and round")
    args = ap.parse_args()

    import torch
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

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, device=dev, generator=gen) * scale

    def p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    layers = []  # (name, callable, flops)
    for lvl in (4, 5, 6):
        x, w, o = rnd(n[lvl], 512), rnd(27, 512, 512, scale=512 ** -0.5 / 5), torch.empty(n[lvl], 512, device=dev)
        macs = C.c_double()

        def f(x=x, w=w, o=o, lvl=lvl, macs=macs):
            check(L.scn_submanifold_convolution_forward(h, l3(sizes[lvl]), l3([3, 3, 3]), p(x), p(o), p(w), None, 512, 512, C.byref(macs), None, 0, None, None))
        f()
        torch.cuda.synchronize()
        layers.append((f"subm 512->512 3^3 level {lvl} ({n[lvl]} sites)", f, 2 * macs.value))
    x, w, o = rnd(n[3], 256), rnd(8, 256, 512, scale=0.02), torch.empty(n[4], 512, device=dev)
    macs4 = C.c_double()

    def fs():
        check(L.scn_convolution_forward(h, l3(sizes[3]), l3(sizes[4]), l3([2, 2, 2]), l3([2, 2, 2]), p(x), p(o), p(w), None, 256, 512, C.byref(macs4), None, 0, None, None))
    fs()
    torch.cuda.synchronize()
    layers.append((f"conv 256->512 2^3/2 level 3->4 ({n[3]} -> {n[4]} sites)", fs, 2 * macs4.value))
    for lvl in (1, 2, 3):
        xc, w, y, wl = rnd(n[lvl + 1], 288), rnd(8, 288, 288, scale=0.03), rnd(n[lvl], 288), rnd(288, 288, scale=0.03)
        y16 = y.to(torch.bfloat16)
        o = torch.empty(n[lvl], 288, device=dev)
        macs = C.c_double()

        def fd(xc=xc, w=w, y=y, y16=y16, wl=wl, o=o, lvl=lvl, macs=macs):
            mode = L.scn_get_math_mode()
            check(L.scn_fuse_next_lateral(p(y), p(y16 if mode == 2 else y.half() if mode == 5 else None), p(wl), 0, 288, n[lvl]))
            check(L.scn_deconvolution_forward(h, l3(sizes[lvl + 1]), l3(sizes[lvl]), l3([2, 2, 2]), l3([2, 2, 2]), p(xc), p(o), p(w), None, 288, 288,
                                              C.byref(macs), None, 0, None, None))
            took_l, took_s = C.c_int(), C.c_int()
            check(L.scn_fuse_result(C.byref(took_l), C.byref(took_s)))
            if not took_l.value:  # (the CUDA-core path: the lateral as its own 1x1x1 product and add, as the program runs it)
                stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                t = torch.empty_like(o)
                check(L.scn_network_in_network_forward(p(y), p(t), p(wl), None, n[lvl], 288, 288, None, stream, None, 0))
                o.add_(t)
        fd()
        torch.cuda.synchronize()
        layers.append((f"deconv 288->288 2^3/2 + lateral 288 level {lvl + 1}->{lvl} ({n[lvl]} sites)", fd, 2 * macs.value + 2.0 * n[lvl] * 288 * 288))

    order = ["bf16", "fp16", "tf32", "tf32x3", "fp32"]
    times = {name: {m: [] for m in order} for name, _, _ in layers}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(args.rounds):
        for m in order:
            check(L.scn_set_math_mode(MODES[m]))
            for name, f, _ in layers:
                f()  # (weight images of this mode)
                tot = 0.0
                for _ in range(args.reps):
                    flush.zero_()
                    ev[0].record()
                    f()
                    ev[1].record()
                    ev[1].synchronize()
                    tot += ev[0].elapsed_time(ev[1])
                times[name][m].append(tot / args.reps)
    check(L.scn_set_math_mode(0))
    per_layer = []
    for name, _, flops in layers:
        row = {"layer": name, "gflop": round(flops / 1e9, 2)}
        for m in order:
            t = med(times[name][m])
            row[m] = {"ms": round(t, 4), "tflops": round(flops / t / 1e9, 1), "share_of_bf16_peak": round(flops / t * 1e3 / BF16_PEAK, 4)}
        row["bf16_speedup_vs_fp32"] = round(row["fp32"]["ms"] / row["bf16"]["ms"], 2)
        per_layer.append(row)

    # ---------------- widened FPN_Net on B470: replayed forward and replayed training step per mode
    cfg = dict(scn.sw4c_fpn432_config(), nPlanesF=[32, 64, 64, 128, 320, 320, 512, 512, 512], nPlaneM=288, track_running_stats=True)
    coords = torch.from_numpy(coords_np)
    feats = torch.from_numpy(fpn_util.features_for(coords_np)).to(dev)
    net_modes = ["bf16", "fp16", "tf32", "tf32x3", "fp32"]
    fwd = {m: [] for m in net_modes}
    trn = {m: [] for m in net_modes}
    nets = {}
    for m in net_modes:
        scn.set_math_mode(m)
        net = scn.FPN_Net(**cfg)
        net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
        ev_net = net.cuda().eval()
        tr_net = scn.FPN_Net(**cfg)
        tr_net.load_state_dict(fpn_util.deterministic_state(tr_net, seed=1))
        tr_net = tr_net.cuda().train()
        nets[m] = (ev_net, tr_net)
        for _ in range(2):  # record, replay once
            with torch.no_grad():
                ev_net([coords, feats])
            rpn, roi = tr_net([coords, feats])
            sum((t.features ** 2).mean() for t in rpn + roi).backward()
        torch.cuda.synchronize()
    for _ in range(args.rounds):
        for m in net_modes:
            scn.set_math_mode(m)
            ev_net, tr_net = nets[m]
            tot = 0.0
            for _ in range(args.steps):
                flush.zero_()
                ev[0].record()
                with torch.no_grad():
                    ev_net([coords, feats])
                ev[1].record()
                ev[1].synchronize()
                tot += ev[0].elapsed_time(ev[1])
            fwd[m].append(tot / args.steps)
            tot = 0.0
            for _ in range(args.train_steps):
                tr_net.zero_grad(set_to_none=True)
                flush.zero_()
                ev[0].record()
                rpn, roi = tr_net([coords, feats])
                sum((t.features ** 2).mean() for t in rpn + roi).backward()
                ev[1].record()
                ev[1].synchronize()
                tot += ev[0].elapsed_time(ev[1])
            trn[m].append(tot / args.train_steps)
    scn.set_math_mode("fp32")
    name, power, clock = card()
    print(json.dumps({"metric": "wide_channel_cost", "card": name, "power_limit": power, "max_sm_clock": clock, "rounds": args.rounds,
                      "sites_per_level": n, "layers": per_layer,
                      "wide_fpn_forward_ms": {m: round(med(fwd[m]), 3) for m in net_modes},
                      "wide_fpn_train_step_ms": {m: round(med(trn[m]), 3) for m in net_modes},
                      "rounds_forward_ms": {m: [round(v, 3) for v in fwd[m]] for m in net_modes},
                      "rounds_train_step_ms": {m: [round(v, 3) for v in trn[m]] for m in net_modes}}))


if __name__ == "__main__":
    main()
