#!/usr/bin/env python
"""Bidirectional flow: one RAFT.forward_backward call against two RAFT.forward calls (l->r, then r->l).

Workload = bench.py's headline: raft-things, 1 pair, 436x1024, 32 iterations, seeded weights and frames resident in HBM,
L2 overwritten (256 MiB write) before every timed step.  The two arms alternate in rounds on two models with the same
weights (each keeps its own graph).  Also times rb_flow_consistency alone with CUDA events over many back-to-back
launches (its 7 MB of flows stay L2-resident there) and checks that the halves equal the forward calls bit for bit.
Prints one JSON line, with the GPU name and power limit read from nvidia-smi (query only).

    python tools/bidir_times.py [--steps 20] [--rounds 3] [--warmup 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "raft-tf_b200"))

import torch  # noqa: E402

H, W, ITERS = 436, 1024, 32


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power = (x.strip() for x in q.split(","))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kernel-reps", type=int, default=500)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bidir_times.py needs a CUDA device")
    from types import SimpleNamespace
    from raft_b200 import capi, synth
    from networks.RAFT import RAFT

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_info(torch.cuda.current_device())
    params = synth.make_weights(False)
    uni = RAFT((H, W, 3), SimpleNamespace(small=False), iters=ITERS, device=dev).load(params)
    bi = RAFT((H, W, 3), SimpleNamespace(small=False), iters=ITERS, device=dev).load(params)
    l_np, r_np = synth.make_batch(1, H, W)
    l, r = torch.from_numpy(l_np).to(dev), torch.from_numpy(r_np).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def two_forward():
        return uni.forward(l, r), uni.forward(r, l)

    def forward_backward():
        return bi.forward_backward(l, r)

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for a, b in evs:
            flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / 1e3

    for _ in range(args.warmup):
        fw, bw = two_forward()
        out = forward_backward()
    exact = torch.equal(out[0], fw) and torch.equal(out[1], bw)
    rate_two, rate_fb = [], []
    for _ in range(args.rounds):  # alternate the arms: other work on the host moves both alike
        rate_two.append(args.steps / timed(two_forward, args.steps))
        rate_fb.append(args.steps / timed(forward_backward, args.steps))

    eng = bi.engine()
    lib, st = capi.lib, capi.stream()
    flow, occ = eng.flow_up, eng.occ

    def consistency():
        capi.check(lib.rb_flow_consistency(capi.ptr(flow[:1]), capi.ptr(flow[1:]), capi.ptr(occ[:1]), capi.ptr(occ[1:]),
                                           1, H, W, 1.0, 0.01, 0.5, st))
    for _ in range(10):
        consistency()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(args.kernel_reps):
        consistency()
    b.record()
    torch.cuda.synchronize()
    t_kernel_us = a.elapsed_time(b) * 1e3 / args.kernel_reps

    med_two, med_fb = statistics.median(rate_two), statistics.median(rate_fb)
    print(json.dumps({
        "workload": f"raft-things 1 pair {H}x{W} (padded 440x1024), {ITERS} iters, frames resident, L2 overwritten "
                    "between steps; a step = the flow in both directions",
        "two_forward_pairs_per_s": round(med_two, 2),
        "forward_backward_pairs_per_s": round(med_fb, 2),
        "speedup": round(med_fb / med_two, 3),
        "rounds": {"two_forward": [round(x, 2) for x in rate_two], "forward_backward": [round(x, 2) for x in rate_fb]},
        "steps_per_round": args.steps,
        "flow_consistency_us": round(t_kernel_us, 2),
        "flow_consistency_note": f"mean of {args.kernel_reps} back-to-back launches, both directions at 436x1024, "
                                 "flows L2-resident",
        "halves_bit_exact": exact,
        "launches": {"forward": uni.engine().launches_per_forward(), "forward_backward": eng.launches_per_forward()},
        "gpu": name, "power_limit": power,
    }), flush=True)


if __name__ == "__main__":
    main()
