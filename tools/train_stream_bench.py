"""What streaming training steps gains (FPN_Net.prefetch in train mode, DESIGN.md section 5 "Streaming"), in one process.

Workload: BASELINE.json config 5 -- the 6c_fpn4321 backbone, one B470-class synthetic building per step (two buildings, seeds 0 and
1, alternating), bf16 mode, replayed training step (one autograd node), one GPU, no all-reduce, loss = sum of squares of the maps,
host coordinates in page-locked memory and device features as in bench.py.  After every step the host synchronises (as a loop that
reads its loss does) and the L2 is overwritten (outside the timed region).  Four modes alternate step block by step block inside
every round, medians over the rounds:

  * plain:            no prefetch; the backward pass builds its rule lists on demand (the default for unprepared steps)
  * plain_lists:      no prefetch; rule lists hinted behind the step's own plans (SCN_TRAIN_LISTS_AHEAD=2)
  * prefetch:         the next step prepared (FPN_Net.prefetch) right after the current forward is queued, before its backward,
                      with its rule lists ahead (the default for prepared steps)
  * prefetch_nolists: the same, lists built on demand (SCN_TRAIN_LISTS_AHEAD=0)

Reported per mode: step time, forward time (step start to loss) and backward time (device events), and -- from a separate
torch.profiler run of a few steps per mode -- the time from the step's start on the host to the start of its first convolution
kernel on the device.  Prints one JSON line with the card's name, power limit and maximum SM clock read in the same run.

    python tools/train_stream_bench.py [--steps 8] [--rounds 3] [--warmup 3] [--profile-steps 4]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True

MODES = ("plain", "plain_lists", "prefetch", "prefetch_nolists")
LISTS_AHEAD = {"plain": "1", "plain_lists": "2", "prefetch": "1", "prefetch_nolists": "0"}  # SCN_TRAIN_LISTS_AHEAD
CONV = re.compile(r"conv_plan_(tc|simt)|conv_list_simt")


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
    ap.add_argument("--steps", type=int, default=8, help="timed steps per round and mode")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile-steps", type=int, default=4, help="profiled steps per mode (time to the first convolution)")
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
    data = []
    for seed in (0, 1):
        c = synthetic.building_coords(seed=seed)
        data.append((torch.from_numpy(c).pin_memory(), torch.from_numpy(fpn_util.features_for(c)).to(dev)))
    scn.set_math_mode("bf16")
    net = scn.FPN_Net(**scn.c6_fpn4321_config())
    net.load_state_dict(fpn_util.deterministic_state(net, seed=1))
    net = net.to(dev).train()
    params = [p for p in net.parameters() if p.requires_grad]
    state = {"i": 0}

    def lists_ahead(mode):
        os.environ["SCN_TRAIN_LISTS_AHEAD"] = LISTS_AHEAD[mode]

    def step(mode, ev=None):
        """one training step on the next building; in the prefetch modes the following one is prepared behind its forward"""
        c, f = data[state["i"] % 2]
        nxt = data[(state["i"] + 1) % 2][0]
        state["i"] += 1
        for p in params:
            p.grad = None
        if ev:
            ev[0].record()
        with torch.profiler.record_function("train_step"):
            rpn, roi = net([c, f])
            loss = sum((m.features ** 2).sum() for m in rpn + roi)
            if ev:
                ev[1].record()
            if mode.startswith("prefetch"):
                assert net.prefetch(nxt)
            loss.backward()
        if ev:
            ev[2].record()
        torch.cuda.synchronize()
        flush.fill_(1)
        torch.cuda.synchronize()

    def start(mode):
        """a block of steps of `mode` begins: its first step is prepared like every later one"""
        lists_ahead(mode)
        net.__dict__.pop("_prefetched_train", None)
        net.__dict__["_program_train"].drop_prepared()
        if mode.startswith("prefetch"):
            assert net.prefetch(data[state["i"] % 2][0])

    step("plain")  # records the training program
    prep0 = lib().scn_debug_counter(20)
    times = {m: {"step": [], "fwd": [], "bwd": []} for m in MODES}
    rules_found = {m: 0 for m in MODES}
    for r in range(args.rounds):
        for mode in MODES:
            start(mode)
            for _ in range(args.warmup if r == 0 else 1):
                step(mode)
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
            r0 = lib().scn_debug_counter(19)
            for ev in evs:
                step(mode, ev)
            rules_found[mode] += lib().scn_debug_counter(19) - r0
            n = len(evs)
            times[mode]["step"].append(sum(e[0].elapsed_time(e[2]) for e in evs) / n)
            times[mode]["fwd"].append(sum(e[0].elapsed_time(e[1]) for e in evs) / n)
            times[mode]["bwd"].append(sum(e[1].elapsed_time(e[2]) for e in evs) / n)
    prepared_runs = lib().scn_debug_counter(20) - prep0

    # time from the step's start on the host to its first convolution kernel on the device, from a profiler trace (run of its own)
    first_conv = {}
    with tempfile.TemporaryDirectory() as tmp:
        for mode in MODES:
            start(mode)
            step(mode)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(args.profile_steps):
                    step(mode)
            path = os.path.join(tmp, mode + ".json")
            prof.export_chrome_trace(path)
            ev = json.load(open(path))["traceEvents"]
            marks = sorted(e["ts"] for e in ev if e.get("name") == "train_step" and e.get("cat") == "user_annotation")
            convs = sorted(e["ts"] for e in ev if e.get("cat") == "kernel" and CONV.search(e.get("name", "")))
            gaps = [min(t for t in convs if t >= m) - m for m in marks if any(t >= m for t in convs)]
            first_conv[mode] = med(gaps) / 1e3 if gaps else None
    os.environ.pop("SCN_TRAIN_LISTS_AHEAD", None)
    scn.set_math_mode("fp32")

    name, power, clock = card()
    result = {"metric": "train_stream", "unit": "ms",
              "step_ms": {m: med(times[m]["step"]) for m in MODES},
              "forward_ms": {m: med(times[m]["fwd"]) for m in MODES},
              "backward_ms": {m: med(times[m]["bwd"]) for m in MODES},
              "first_conv_ms": first_conv,
              "rounds_ms": times,
              "rule_lists_found_built": rules_found, "prepared_runs": prepared_runs,
              "gpu": name, "power_limit": power, "max_sm_clock": clock,
              "workload": "BASELINE.json config 5: 6c_fpn4321 replayed training step, B470-class buildings (seeds 0, 1 alternating), bf16, one GPU, "
                          "no all-reduce; host synchronised and L2 overwritten after every step (outside the timed region)",
              "steps": args.steps, "rounds": args.rounds, "warmup": args.warmup, "profile_steps": args.profile_steps}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
