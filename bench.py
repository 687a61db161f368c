#!/usr/bin/env python
"""bench.py -- frame-pairs/s of the RAFT recurrent-inference path (BASELINE.json metric).

Workload (N GPUs, weak scaling): BASELINE config[1] per GPU -- raft-things, 1 frame pair per GPU,
436x1024 (replicate-padded to 440x1024, SURVEY 8(d)), 32 iterations, synthetic frames, seeded
random weights in the reference's npz naming (no network: neither Sintel nor the Drive weights).
A "step" = one forward pass (encoders + correlation build + 32 x (lookup, update block) + convex
upsampling) over the batch.

  value  : pairs/s with the frames already resident in HBM (CUDA events, max over ranks)
  e2e    : pairs/s through the public API (networks.RAFT.RAFT.forward) with PINNED HOST frames:
           H2D of both frames and D2H of the flow inside the timed region, every step
  roofline        : the update-block convolutions (dominant: ~97% of hot-path FLOPs), tensor bound
  roofline_lookup : the correlation-lookup kernel (the metric's namesake), HBM bound (B=1 cold / L2-warm, B=8)
  roofline_corr   : rb_corr_build (volume + pooled levels), HBM side and tensor side
  other_configs   : BASELINE configs 3-5, batch-sharded over the launched GPUs, NCCL all_gather inside the e2e span
  cpu_baseline    : the CPU oracle (torch fp32 restatement of the reference; TF is not installable)
                    timed on the host cores of the same box

--impl reference times that same CPU restatement as the reference arm (oracle/ is executed only
there and in cpu_baseline).
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "raft-tf_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

H_IMG, W_IMG, ITERS, SMALL = 436, 1024, 32, False
H_PAD, W_PAD = 440, 1024
METRIC = "frame-pairs/sec @ 436x1024, 32 iters (raft-things)"
# algorithmic work per sample (SURVEY 8(d)): update block MAC/px/iter, lookup bytes/px/iter
UPDATE_MAC_PER_PX = 2675968
LOOKUP_BYTES_PER_PX = 2904  # N*[4*((2r+2)^2*4 + (2r+1)^2*4) + 8], r=4, fp32 volume, fp32-equivalent output


def workload(b_per_gpu=1):
    """config.workload -- the SAME string in both arms (the driver compares them)."""
    return f"raft-things B={b_per_gpu}/GPU {H_IMG}x{W_IMG} (padded {H_PAD}x{W_PAD}) {ITERS} iters"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf=p["bf16_tflops"], tf_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.kill)  # never leave the sampler running, also when the benchmark fails before stop()
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark(self):
        """Number of samples received so far (brackets the timed region inside a longer sampling run)."""
        return len(self.lines)

    def stop(self, first=0, last=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines[first:last]:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def effective_cores():
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:  # cgroup v2 quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def cpu_sample(threads):
    """One step of the workload on the host CPU: the full 440x1024 pair through encoders, correlation pyramid, ALL 32
    iterations and the convex upsampling of the CPU oracle (torch fp32 restatement of the reference; nothing is
    extrapolated).  Returns (seconds per pair, description, [1,440,1024,2] flow)."""
    from oracle.raft_oracle import RAFTOracle, upsample_flow
    from raft_b200 import synth
    torch.set_num_threads(threads)
    params = synth.make_weights(SMALL)
    l, r = synth.make_batch(1, H_PAD, W_PAD)
    m = RAFTOracle(params, small=SMALL, iters=ITERS)
    t0 = time.perf_counter()
    st = m.prepare(torch.from_numpy(l), torch.from_numpy(r))
    t1 = time.perf_counter()
    net, mask, c1 = m.iterate(st)
    flow = upsample_flow(c1 - st["coords0"], mask)
    t2 = time.perf_counter()
    desc = (f"1 frame pair {H_PAD}x{W_PAD}, all {ITERS} iterations measured (encoders + volume {t1 - t0:.2f}s, iterations + "
            f"upsampling {t2 - t1:.2f}s); torch-CPU fp32 oracle, {threads} threads")
    return t2 - t0, desc, flow


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each array as out_dir/<name>.npy (float32) so that two builds run with the same arguments
    can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32, copy=False))


def run_reference(args, rank, world):
    """Reference arm: the reference's algorithm on the host CPU (oracle port; the TF original cannot be
    installed here -- no network, no wheels).  Rank 0 only."""
    if rank != 0:
        return
    cores = effective_cores()
    threads = min(cores, 32)  # torch-CPU conv scaling is flat beyond ~32 threads at these sizes
    for _ in range(args.warmup):
        cpu_sample(threads)
    ts = []
    desc = ""
    for _ in range(args.steps):
        t, desc, flow = cpu_sample(threads)
        ts.append(t)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"flow": flow})
    dt = sum(ts)
    v = args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload(1), "global_batch": 1,
                       "note": "CPU restatement of gonglixue/RAFT-tf (TensorFlow/tensorpack not installable offline); "
                               "one process on the host cores whatever --gpus says"},
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def other_configs(args, rank, world, dev, timed, dist):
    """BASELINE.json configs[2..4] on the launched GPUs, batch-sharded (SURVEY 8(e)): every rank runs its slice of the
    global batch, the [B/G,H,W,2] flows are all_gathered over NCCL so that each rank holds the full result.

      config3  raft-things  B=8          540x960 (-> 544x960), 32 it   -- single-GPU config: N=1 only
      config4  raft-things  B=4 per GPU  436x1024, 32 it               -- 32 pairs over 8 GPUs
      config5  raft-small   B=8 per GPU  768x1024, 20 it               -- 64 pairs over 8 GPUs

    value = global pairs/s with frames resident (max over ranks); e2e = pinned-host frames in, H2D + forward + NCCL
    all_gather + D2H of this rank's shard inside the timed span; gather_us = the all_gather alone (CUDA events)."""
    from types import SimpleNamespace
    from raft_b200 import synth
    from networks.RAFT import RAFT
    specs = [("config4", False, 4, 436, 1024, 32), ("config5", True, 8, 768, 1024, 20)]
    if world == 1:
        specs.insert(0, ("config3", False, 8, 540, 960, 32))
    out = {}
    steps = args.steps
    for name, small, b, H, W, iters in specs:
        try:
            m = RAFT((H, W, 3), SimpleNamespace(small=small), iters=iters, batch=b, device=dev).load(synth.make_weights(small))
            l_np, r_np = synth.make_batch(b, H, W, seed0=2000 + rank * b)
            lh, rh = torch.from_numpy(l_np).pin_memory(), torch.from_numpy(r_np).pin_memory()
            ld, rd = lh.to(dev), rh.to(dev)
            oh = torch.empty(b, H, W, 2, dtype=torch.float32).pin_memory()
            full = torch.empty(world * b, H, W, 2, dtype=torch.float32, device=dev)
            gev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

            def gather(flow):
                if world > 1:
                    gev[0].record()
                    dist.all_gather_into_tensor(full, flow.contiguous())
                    gev[1].record()

            def res():
                gather(m.engine().forward(ld, rd))

            def e2e():
                flow = m.engine().forward(lh, rh)
                gather(flow)
                oh.copy_(flow, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            for _ in range(2):
                res(); e2e()
            t_r, t_e = timed(res, steps), timed(e2e, steps)
            pairs = b * world * steps
            g_us = None
            if world > 1:
                torch.cuda.synchronize()
                g_us = gev[0].elapsed_time(gev[1]) * 1e3
            out[name] = {"workload": f"raft-{'small' if small else 'things'} B={b}/GPU {H}x{W} {iters} iters",
                         "global_batch": b * world, "value": pairs / t_r, "unit": "pairs/s", "ms_per_step": t_r / steps * 1e3,
                         "e2e": {"value": pairs / t_e, "h2d_bytes_per_step": int(lh.numel() * 8), "d2h_bytes_per_step": int(oh.numel() * 4),
                                 "ms_per_step": t_e / steps * 1e3},
                         "gather_us": g_us, "gather_bytes_per_rank": int(b * H * W * 8) if world > 1 else 0, "steps": steps}
            del m, ld, rd, full
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001 -- an extra: never lose the headline line for it
            out[name] = {"error": str(e)[:300]}
    return out


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the other BASELINE configs (other_configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the flow of the last timed headline step to DIR/flow.npy "
                         "(float32; DIR/flow_rank<r>.npy for ranks > 0; the leading samples of the batch that fit "
                         "in 64 MiB over all ranks)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from types import SimpleNamespace
    from raft_b200 import capi, synth
    from networks.RAFT import RAFT

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch_per_gpu
    params = synth.make_weights(SMALL)
    model = RAFT((H_IMG, W_IMG, 3), SimpleNamespace(small=SMALL), iters=ITERS, batch=B, device=dev).load(params)
    l_np, r_np = synth.make_batch(B, H_IMG, W_IMG, seed0=1000 + rank * B)
    l_host = torch.from_numpy(l_np).pin_memory()
    r_host = torch.from_numpy(r_np).pin_memory()
    l_dev, r_dev = l_host.to(dev), r_host.to(dev)
    out_host = torch.empty(B, H_IMG, W_IMG, 2, dtype=torch.float32).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps, L2 flushed between steps (flush excluded from the timed spans); returns seconds (max over ranks)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for a, b in evs:
            flush.zero_()
            a.record()
            fn()
            b.record()
        barrier()
        t = sum(a.elapsed_time(b) for a, b in evs) / 1e3
        if world > 1:
            tt = torch.tensor([t], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt.item())
        return t

    last = {}

    def step_resident():
        last["flow"] = model.forward(l_dev, r_dev)  # a fresh tensor per call (RAFT.forward): what a caller receives

    def step_e2e():
        flow = model.forward(l_host, r_host)  # H2D of both frames inside
        out_host.copy_(flow, non_blocking=True)  # D2H of the result
        torch.cuda.current_stream().synchronize()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()  # nvidia-smi needs ~0.1 s to deliver its first sample: start it before the warm-up
    for _ in range(args.warmup):
        step_resident()
    eng = model.engine()
    launches_per_fwd = eng.launches_per_forward()
    m0 = clocks.mark()
    t_res = timed(step_resident, args.steps)
    flow_last = last["flow"]  # output of the last timed step (the untimed steps below must not replace it)
    m1 = clocks.mark()
    clk = None
    if rank == 0:
        extended = False
        t_wait = time.time()
        while clocks.mark() - m0 < 3 and time.time() - t_wait < 3.0 and clocks.proc is not None:
            # timed region shorter than the sampling period: keep the SAME load running (untimed) until 3 samples exist
            step_resident()
            extended = True
        if extended:
            torch.cuda.synchronize()
            m1 = clocks.mark()
        clk = clocks.stop(m0, max(m1, m0 + 1))
        clk["sampled"] = "timed region + identical untimed steps" if extended else "timed region"
    for _ in range(2):
        step_e2e()
    t_e2e = timed(step_e2e, args.steps)

    # ---- per-kernel rooflines, measured live with CUDA events on the launching stream ----
    pk = peaks()
    h, w, s = eng.h, eng.w, int(SMALL)
    npix = B * h * w
    lib = capi.lib

    def ev_time(fn, reps=10, flush_l2=True):
        """Device time of fn() per call: `reps` x (L2 flush; fn) replayed from one CUDA graph minus the same graph
        without fn -- event timing of eager launches would measure the host launch latency for ~5 us kernels."""
        def build(with_fn, n=reps):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(n):
                    if flush_l2:
                        flush.zero_()
                    if with_fn:
                        fn()
            return g
        fn(); torch.cuda.synchronize()
        # baseline: the same graph without fn; without the flush that graph would be empty, so difference 2*reps against reps
        g1, g0 = (build(True), build(False)) if flush_l2 else (build(True, 2 * reps), build(True, reps))
        def run(g):
            ts = []
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); g.replay(); b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b) / 1e3)
            return statistics.median(ts)
        return max(run(g1) - run(g0), 1e-9) / reps

    c1 = eng.coords1.clone()
    t_upd = ev_time(lambda: capi.check(lib.rb_update_step(s, capi.ptr(eng.blob), capi.ptr(eng.ws), capi.ptr(c1), None, None,
                                                           B, h, w, capi.stream())))
    look = lambda: capi.check(lib.rb_update_lookup(s, capi.ptr(eng.ws), capi.ptr(eng.pyramid), capi.ptr(eng.coords1),  # noqa: E731
                                                   B, h, w, capi.stream()))
    t_look = ev_time(look)
    t_look_warm = ev_time(look, flush_l2=False)
    upd_flops = 2.0 * npix * UPDATE_MAC_PER_PX
    look_bytes = float(npix * LOOKUP_BYTES_PER_PX)
    roof = {"kernel": "rb_update_step: 10 tcgen05 convs (conv_tc_kernel, PDL-chained) + flow_conv7_kernel", "bound": "tensor",
            "achieved": upd_flops / t_upd / 1e12, "peak": pk["tf"], "unit": "TFLOP/s",
            "frac": upd_flops / t_upd / 1e12 / pk["tf"], "traffic": None, "peak_source": pk["src"],
            "note": "algorithmic fp32-equivalent FLOPs; each product costs 3 fp16 MMAs (hi/lo split), so frac <= 1/3 by design",
            "us_per_launch_group": t_upd * 1e6}
    roof_l = {"kernel": "corr_lookup_kernel<4,split>", "bound": "hbm", "achieved": look_bytes / t_look / 1e9,
              "peak": pk["hbm"], "unit": "GB/s", "frac": look_bytes / t_look / 1e9 / pk["hbm"], "traffic": 35.45e6 * B,
              "traffic_note": "ncu --set full (profiles/r02_lookup_ncu_full.txt): dram read 35.41 MB + write 0.04 MB per cold launch (TMA boxes of 16 columns x 10 rows: whole 64-byte granules)",
              "peak_source": pk["src"], "us_per_launch": t_look * 1e6,
              "l2_warm": {"us_per_launch": t_look_warm * 1e6, "achieved": look_bytes / t_look_warm / 1e9,
                          "note": "same launch without the L2 flush: at B=1 the ~25 MB of patches around the current flow stay L2-resident between iterations"}}

    # the same kernel on a batch whose touched footprint exceeds L2 (8 samples, random pyramid): the HBM-bound regime
    try:
        B8 = 8
        pyr8 = torch.randn(capi.size_query(lib.rb_corr_pyramid_bytes, B8, h, w) // 4, device=dev)
        ws8 = torch.zeros(capi.size_query(lib.rb_update_workspace_bytes, s, B8, h, w), dtype=torch.uint8, device=dev)
        g8 = torch.stack(torch.meshgrid(torch.arange(w, device=dev), torch.arange(h, device=dev), indexing="xy"), -1).float()
        c8 = (g8[None] + torch.rand(B8, h, w, 2, device=dev) * 16 - 8).contiguous()
        t8 = ev_time(lambda: capi.check(lib.rb_update_lookup(s, capi.ptr(ws8), capi.ptr(pyr8), capi.ptr(c8), B8, h, w, capi.stream())))
        roof_l["batch8"] = {"us_per_launch": t8 * 1e6, "achieved": B8 * h * w * LOOKUP_BYTES_PER_PX / t8 / 1e9,
                            "frac": B8 * h * w * LOOKUP_BYTES_PER_PX / t8 / 1e9 / pk["hbm"],
                            "traffic": 340.6e6,
                            "traffic_note": "ncu --set full (profiles/r02_lookup_ncu_full.txt): dram read 285.9 MB + write 54.6 MB in 67.0 us = 5.08 TB/s = 0.77 of the copy peak on REAL traffic (64-byte DRAM granules around 40-44-byte row segments)",
                            "note": "B=8 x 440x1024 grid, N(0,1) pyramid (2.1 GB), coords = grid + U(-8,8), L2 flushed"}
        del pyr8, ws8
    except Exception as e:  # noqa: BLE001 -- an extra, never fail the bench line for it
        roof_l["batch8"] = {"error": str(e)[:200]}

    # ---- correlation build (A1): four tcgen05 GEMMs + operand split / pooling passes; the 261 MB fp32 volume write is its
    # HBM side, 2*N^2*C*(1+1/4+1/16+1/64) its tensor side (SURVEY 8(d): "balanced; report both")
    t_corr = ev_time(lambda: capi.check(lib.rb_corr_build(capi.ptr(eng.fmap1), capi.ptr(eng.fmap2), capi.ptr(eng.pyramid), B, h, w,
                                                          eng.fdim, capi.ptr(eng.corr_ws), eng.cws_bytes, capi.stream())), reps=5)
    N1 = h * w
    lvl_elems = sum((h >> l) * (w >> l) for l in range(4))
    corr_bytes = float(B * (2 * N1 * eng.fdim * 4 + N1 * lvl_elems * 4))
    corr_flops = 2.0 * B * N1 * lvl_elems * eng.fdim
    roof_c = {"kernel": "rb_corr_build: conv_tc_kernel x4 (volume + 3 pooled levels by linearity) + split/pool passes",
              "bound": "hbm", "achieved": corr_bytes / t_corr / 1e9, "peak": pk["hbm"], "unit": "GB/s",
              "frac": corr_bytes / t_corr / 1e9 / pk["hbm"], "traffic": 158.6e6 * B,
              "traffic_note": "ncu --set full (profiles/r02_corr_ncu_full.txt), level-0 GEMM: dram read 14.5 MB + write 144.1 MB inside the kernel (the rest of the 198 MB it stores is still in L2 when it ends)",
              "peak_source": pk["src"],
              "us_per_launch_group": t_corr * 1e6, "algorithmic_bytes": corr_bytes,
              "tensor": {"achieved": corr_flops / t_corr / 1e12, "unit": "TFLOP/s (fp32-equivalent; 3 fp16 MMAs per product)",
                         "frac": corr_flops / t_corr / 1e12 / pk["tf"]}}

    # ---- e2e with uint8 host frames (what cv2.imdecode yields; /255 on the GPU): 4x fewer H2D bytes ----
    l8 = torch.from_numpy(np.round(l_np * 255.0).astype(np.uint8)).pin_memory()
    r8 = torch.from_numpy(np.round(r_np * 255.0).astype(np.uint8)).pin_memory()

    def step_e2e_u8():
        flow = model.forward(l8, r8)
        out_host.copy_(flow, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    for _ in range(2):
        step_e2e_u8()
    t_e2e_u8 = timed(step_e2e_u8, args.steps)

    # ---- the other BASELINE.json configurations, batch-sharded as SURVEY 8(e) specifies ----
    others = {}
    if not args.headline_only:
        others = other_configs(args, rank, world, dev, timed, dist)

    if args.dump_outputs:
        keep = max(1, (64 << 20) // world // (flow_last[0].numel() * 4))  # <= 64 MiB over all ranks: leading samples
        dump_outputs(args.dump_outputs, {"flow" if rank == 0 else f"flow_rank{rank}": flow_last[:keep]})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = min(effective_cores(), 32)
        cpu_sample(threads)  # warm-up (page-in, oneDNN primitive caches)
        tc, desc, _ = cpu_sample(threads)
        cpu = {"value": 1.0 / tc, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": desc}

    if rank == 0:
        pairs = B * world * args.steps
        in_bytes = int(l_host.numel() * 4 * 2)
        line = {"metric": METRIC, "value": pairs / t_res, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 (fp16 hi/lo split operands, fp32 accumulate)",
                "data": "synthetic",
                "config": {"workload": workload(B), "global_batch": B * world, "parallelism": f"dp{world}",
                           "l2": "flushed between steps (256 MiB write)", "weights": "seeded random (synth.make_weights)"},
                "e2e": {"value": pairs / t_e2e, "unit": "pairs/s", "h2d_bytes_per_step": in_bytes,
                        "d2h_bytes_per_step": int(out_host.numel() * 4), "ms_per_step": t_e2e / args.steps * 1e3},
                "gpu_launches": launches_per_fwd * args.steps, "gpu_launches_per_step": launches_per_fwd,
                "roofline": roof, "roofline_lookup": roof_l, "roofline_corr": roof_c, "clocks": clk}
        line["e2e"]["u8_frames"] = {"value": pairs / t_e2e_u8, "unit": "pairs/s", "h2d_bytes_per_step": int(l8.numel() * 2),
                                    "ms_per_step": t_e2e_u8 / args.steps * 1e3,
                                    "note": "same call with uint8 BGR host frames (cv2.imdecode's type); x/255 on the GPU"}
        if others:
            line["other_configs"] = others
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
