#!/usr/bin/env python
"""bench.py -- image-pairs/sec of the UniMatch matching path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config4|config2|config3|config5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step = one `UniMatch.forward` over one batch of synthetic pairs.  Default workload = BASELINE.json configs[3]
(gmflow-scale2-regrefine6, 480x832, 64 pairs over 8 GPUs = 8 pairs per GPU; weak scaling, so N=1 runs 8 pairs); `--workload`
selects configs[1] / [2] / [4] (gmflow-scale1 B=32, gmstereo-scale2 B=16 at 544x960, gmdepth-scale1-regrefine1 at 384x512).
Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM; `e2e`: host pinned buffers in, host result out, copies inside
the timed region.  `--impl reference` times the CPU oracle port of the reference path on the host's physical cores.
`epe_vs_reference` compares pair 0 of the GPU output with the oracle (== reference) and carries its tolerance and a pass flag;
a failing parity check makes the process exit non-zero after printing the line.
`--dump-outputs DIR` writes the prediction of the last timed step (rank 0) as DIR/<flow|disparity|depth>.npy, float32, at
most 64 MB (a larger output is cut to a seeded sample of whole pairs, listed in the JSON line).  Inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "image-pairs/sec @480x832 gmflow-scale2-refine6; EPE vs reference"
# name -> (workload, H, W, pairs per GPU, BASELINE.json configs index, metric string, (mean tol, max tol, unit))
BENCH_WORKLOADS = {
    "config4": ("gmflow-scale2-regrefine6", 480, 832, 8, 3, METRIC, (1e-2, 1e-1, "px EPE")),
    "config2": ("gmflow-scale1", 480, 832, 32, 1, "image-pairs/sec @480x832 gmflow-scale1; EPE vs reference", (1e-2, 1e-1, "px EPE")),
    "config3": ("gmstereo-scale2", 544, 960, 16, 2, "image-pairs/sec @544x960 gmstereo-scale2; l1 disparity vs reference",
                (2e-2, 2e-1, "px |disparity error|")),
    "config5": ("gmdepth-scale1-regrefine1", 384, 512, 8, 4, "image-pairs/sec @384x512 gmdepth-scale1-regrefine1; l1 depth vs reference",
                (1e-4, 1e-3, "|depth error|")),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d["bf16_tflops_sustained"], tflops_burst=d["bf16_tflops"], source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source="fallback")


def physical_cores():
    """Physical core count of the host (SURVEY.md section 8d: the CPU baseline runs on all physical cores, count printed)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    try:
        ids = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip() and phys is not None:
                ids.add((phys, core)); phys = core = None
        if ids:
            return len(ids)
    except OSError:
        pass
    return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_LIMIT = 64 * 10 ** 6               # bytes written by --dump-outputs


def dump_outputs(directory, task, out):
    """Write `out` ([B,2,H,W] flow or [B,H,W] disparity / depth) as float32 .npy under `directory`; above DUMP_LIMIT a
    seeded sample of whole pairs is written instead.  Returns what was written, for the JSON line."""
    import numpy as np
    name = {"flow": "flow", "stereo": "disparity", "depth": "depth"}[task] + ".npy"
    out = out.detach().float().cpu()
    pairs = None
    if out.numel() * 4 > DUMP_LIMIT:
        k = DUMP_LIMIT // (out[0].numel() * 4)
        pairs = torch.randperm(out.shape[0], generator=torch.Generator().manual_seed(0))[:k].sort().values
        out = out[pairs]
        pairs = pairs.tolist()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name), out.numpy())
    return {"dir": os.path.abspath(directory), "files": {name: list(out.shape)}, "pairs": pairs}


def run_oracle_once(sd, cfg, batch, threads, device="cpu"):
    """One forward of the oracle port (the reference's own ATen op sequence, oracle/unimatch_oracle.py)."""
    from oracle import unimatch_oracle as O
    torch.set_num_threads(threads)
    mk = {k: cfg["model"][k] for k in ("num_scales", "upsample_factor", "reg_refine")}
    b = {k: v.to(device) for k, v in batch.items()}
    sdd = sd if device == "cpu" else {k: v.to(device) for k, v in sd.items()}
    if device != "cpu":
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = O.forward(sdd, b["img0"], b["img1"], intrinsics=b.get("intrinsics"), pose=b.get("pose"), **mk, **cfg["call"])["flow_preds"][-1]
    if device != "cpu":
        torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def error_vs(ref, got):
    d = (got - ref).norm(dim=1) if ref.dim() == 4 else (got - ref).abs()
    return d.mean().item(), d.max().item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config4", choices=sorted(BENCH_WORKLOADS))
    ap.add_argument("--pairs-per-gpu", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference-eager-on-this-GPU line (oracle port on cuda, TF32 off)")
    ap.add_argument("--profile", action="store_true", help="1 warm-up + K steps of the resident path only (for ncu launch lists)")
    ap.add_argument("--graph", action="store_true", help="replay the forward as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's prediction as DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncores = physical_cores()

    from unimatch_b200.spec import WORKLOADS
    from unimatch_b200.synthetic import BENCH_WEIGHTS, synthetic_batch, synthetic_state_dict
    wl_name, H, W, ppg, cfg_idx, metric, (tol_mean, tol_max, err_unit) = BENCH_WORKLOADS[args.workload]
    Bp = args.pairs_per_gpu or ppg
    cfg = WORKLOADS[wl_name]
    task = cfg["model"]["task"]
    sd = synthetic_state_dict(seed=326, **BENCH_WEIGHTS, **cfg["model"])
    config = {"workload": "%s %dx%d, %d pairs/GPU (BASELINE configs[%d])" % (wl_name, H, W, Bp, cfg_idx),
              "global_batch": Bp * world, "parallelism": "dp%d (pairs sharded, no data-path collective; NCCL all_gather of outputs off the critical path)" % world,
              "weights": "synthetic seed 326, well-conditioned set %s (same shapes / arithmetic as random init; reference self-noise 2e-5 px, tools/self_noise.py)" % json.dumps(BENCH_WEIGHTS),
              "l2": "per-step working set >> 126 MB L2 (activations of the batch), no flush needed"}
    ARITHMETIC = ("fp32-faithful: tensor-core products as fp16 (hi, lo) split operands (hi*hi + hi*lo + lo*hi, fp32 accumulate), "
                  "everything else fp32 on CUDA cores; no TF32 / BF16 single-pass products")

    # ------------------------------------------------------------------ reference arm: CPU oracle port on host cores
    if args.impl == "reference":
        if rank != 0:
            return
        batch = synthetic_batch(task, 1, H, W, first_index=0)
        budget = 240.0
        t_start = time.perf_counter()
        times = []
        for i in range(args.warmup + args.steps):
            out, dt = run_oracle_once(sd, cfg, batch, ncores)
            if i >= args.warmup or (time.perf_counter() - t_start) > budget:
                times.append(dt)
            if (time.perf_counter() - t_start) > budget and times:
                break
        sec = sum(times) / len(times)
        val = 1.0 / sec
        dumped = {"dump_outputs": dump_outputs(args.dump_outputs, task, out)} if args.dump_outputs else {}
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": len(times), "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": ncores, "host_logical_cpus": os.cpu_count(), "kind": "port",
                             "sample": "1 pair per step, %d timed steps (240 s budget), torch threads = physical cores" % len(times)},
            "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, **dumped}))
        return

    # ------------------------------------------------------------------ our arm
    import torch.distributed as dist
    from unimatch_b200 import UniMatch, ops
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = UniMatch(**cfg["model"]).eval()
    model.load_state_dict(sd, strict=True)
    model = model.to(dev)
    host = synthetic_batch(task, Bp, H, W, first_index=rank * Bp)
    pinned = {k: v.pin_memory() for k, v in host.items()}
    resident = {k: v.to(dev) for k, v in pinned.items()}
    extra_keys = [k for k in host if k not in ("img0", "img1")]             # intrinsics / pose (depth)
    out_shape = (Bp, 2, H, W) if task == "flow" else (Bp, H, W)
    out_host = torch.empty(out_shape, dtype=torch.float32).pin_memory()

    graph, static_out = None, None
    use_graph = args.graph and not args.profile

    def forward_eager(inp):
        return model(inp["img0"], inp["img1"], intrinsics=inp.get("intrinsics"), pose=inp.get("pose"), **cfg["call"])["flow_preds"][-1]

    if use_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                forward_eager(resident)                    # warm-up: lazy inits, cudaFuncSetAttribute, allocator pools, plane caches
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = forward_eager(resident)
        torch.cuda.synchronize()

    def forward(from_host=False):
        if graph is None:
            if not from_host:
                return forward_eager(resident)
            return forward_eager({k: v.to(dev, non_blocking=True) for k, v in pinned.items()})
        if from_host:
            for k in ("img0", "img1"):
                resident[k].copy_(pinned[k], non_blocking=True)
        graph.replay()
        return static_out

    # The only collective is the gather of the predictions (SURVEY.md section 8e).  It is issued asynchronously (NCCL's own
    # stream, ordered after the forward by an event) into one of two buffers and waited for one step later, so a rank never
    # stalls on the slowest rank's step inside the timed loop; everything is drained before the closing event.
    gather_bufs = [torch.empty((world,) + out_shape, device=dev) for _ in range(2)] if world > 1 else None
    local_bufs = [torch.empty(out_shape, device=dev) for _ in range(2)] if world > 1 else None
    pending = [None, None]
    step_no = [0]

    def gather_async(flow):
        if world == 1:
            return
        i = step_no[0] & 1
        if pending[i] is not None:
            pending[i].wait()
        local_bufs[i].copy_(flow)                              # the forward's output buffer is free for the next step
        pending[i] = dist.all_gather_into_tensor(gather_bufs[i].view(-1), local_bufs[i].view(-1), async_op=True)
        step_no[0] += 1

    def gather_drain():
        for i in range(2):
            if pending[i] is not None:
                pending[i].wait()
                pending[i] = None

    last = [None]                                          # the prediction of the latest resident step

    def step_resident():
        flow = forward()
        gather_async(flow)
        last[0] = flow
        return flow

    # End-to-end path: every step's inputs come from pinned host memory and its result goes back to pinned host memory,
    # all inside the timed region.  The copies run on a copy stream, double-buffered (as unimatch_b200.BatchedFlowRunner does
    # for a stream of frames): H2D of step i+1 and D2H of step i-1 overlap the forward of step i.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_in = [{k: torch.empty_like(v) for k, v in resident.items()} for _ in range(2)]
    dev_out = [torch.empty(out_shape, device=dev) for _ in range(2)]
    h2d_done = [None, None]
    d2h_done = [None, None]
    e2e_no = [0]

    def e2e_prefetch(slot):
        with torch.cuda.stream(copy_stream):
            for k in dev_in[slot]:
                dev_in[slot][k].copy_(pinned[k], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        h2d_done[slot] = ev

    def step_e2e():
        main = torch.cuda.current_stream()
        i = e2e_no[0] & 1
        if h2d_done[i] is None:                                # first step: nothing was prefetched yet
            copy_stream.wait_stream(main)
            e2e_prefetch(i)
        main.wait_event(h2d_done[i])
        if graph is None:
            flow = forward_eager(dev_in[i])
        else:
            for k in ("img0", "img1"):
                resident[k].copy_(dev_in[i][k], non_blocking=True)
            graph.replay()
            flow = static_out
        if d2h_done[i] is not None:
            main.wait_event(d2h_done[i])                       # the result of two steps ago has left dev_out[i]
        dev_out[i].copy_(flow, non_blocking=True)              # the forward's output buffer is reused by the next step
        fwd_done = torch.cuda.Event()
        fwd_done.record(main)
        gather_async(dev_out[i])
        copy_stream.wait_event(fwd_done)                       # inputs of slot i^1 were consumed two steps ago; dev_out[i] is ready
        e2e_prefetch(i ^ 1)                                    # next step's inputs
        with torch.cuda.stream(copy_stream):
            out_host.copy_(dev_out[i], non_blocking=True)      # this step's result -> pinned host
            d2h_done[i] = torch.cuda.Event()
            d2h_done[i].record(copy_stream)
        e2e_no[0] += 1
        return flow

    def e2e_drain():
        torch.cuda.current_stream().wait_stream(copy_stream)

    def timed(fn, steps, sample_clocks=False, timer=None, per_step=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        if timer is not None:
            model.kernel_timer = timer
        l0 = ops.launch_count()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        marks[0].record()
        for i in range(steps):
            fn()
            if per_step:
                marks[i + 1].record()
        gather_drain()
        e2e_drain()
        marks[-1].record()
        torch.cuda.synchronize()
        model.kernel_timer = None
        if timer is not None:
            for tag, a, b, fl in timer.pop("_events", []):
                acc = timer.setdefault(tag, [0.0, 0, 0.0])
                acc[0] += a.elapsed_time(b); acc[1] += 1; acc[2] += fl
        if world > 1:
            dist.barrier()
        ms = marks[0].elapsed_time(marks[-1])
        steps_ms = [marks[i].elapsed_time(marks[i + 1]) for i in range(steps)] if per_step else None
        launches = ops.launch_count() - l0
        clocks = sampler.stop() if sampler else None
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches, clocks, (ms, steps_ms)

    if args.profile:
        step_resident()
        ms, launches, _, _ = timed(step_resident, args.steps)
        dumped = {"dump_outputs": dump_outputs(args.dump_outputs, task, last[0])} if args.dump_outputs and rank == 0 else {}
        print(json.dumps({"profile_run": True, "ms_per_step": ms / args.steps, "gpu_launches": launches, **dumped}))
        return
    for _ in range(max(args.warmup, 3)):
        step_resident()
    gather_drain()
    ms, launches_r, clocks, (ms_own, steps_ms) = timed(step_resident, args.steps, sample_clocks=True, per_step=True)
    # copied now: with --graph the later passes replay into the same output buffer
    dumped = dump_outputs(args.dump_outputs, task, last[0]) if args.dump_outputs and rank == 0 else None
    # kernel-level timers and the launch counter live in the eager path: a separate pass (events around every launch group
    # perturb the host side, so this pass is not the one `value` is taken from)
    timer = {}
    ms_timed, launches, _, _ = timed(lambda: forward_eager(resident), args.steps, timer=timer)
    for _ in range(2):
        step_e2e()
    gather_drain()
    e2e_drain()
    h2d_done[0] = h2d_done[1] = None                       # the timed region starts cold: its first step pays its own H2D
    e2e_no[0] = 0
    ms_e2e, _, _, _ = timed(step_e2e, args.steps)
    # gather-only time (all ranks enter together; the wire time of the output exchange)
    gather_ms = None
    if world > 1:
        flow = forward()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            dist.all_gather_into_tensor(gather_bufs[0].view(-1), flow.contiguous().view(-1))
        e1.record()
        torch.cuda.synchronize()
        gather_ms = e0.elapsed_time(e1) / 5
    flow = forward_eager(resident)
    torch.cuda.synchronize()

    total_pairs = Bp * world
    value = total_pairs * args.steps / (ms / 1e3)
    e2e = total_pairs * args.steps / (ms_e2e / 1e3)

    # per-rank step statistics (is the job limited by one slow GPU, by the exchange, or by the host?)
    own = sorted(steps_ms)
    stats = torch.tensor([own[0], own[len(own) // 2], own[-1], ms_own / args.steps], device=dev)
    if world > 1:
        allstats = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(allstats, stats)
    else:
        allstats = [stats]
    rank_stats = [{"rank": r, "step_ms_min": round(s[0].item(), 3), "step_ms_median": round(s[1].item(), 3),
                   "step_ms_max": round(s[2].item(), 3), "mean_ms_per_step": round(s[3].item(), 3)} for r, s in enumerate(allstats)]

    # ---- rooflines: the fused attention kernel (tensor-bound) and the convolution / Linear family (tensor-bound)
    pk = peaks()
    traffic, traffic_detail = None, None
    tp = os.path.join(ROOT, "profiles", "r02_ncu_kernels.json")
    if os.path.exists(tp):                                  # dram bytes per launch from the committed ncu --set full capture
        try:
            items = [d for d in json.load(open(tp)) if "attention" in d.get("label", "")]
            traffic_detail = {d["label"]: d["dram__bytes_read.sum"] + d["dram__bytes_write.sum"] for d in items}
            if traffic_detail:
                traffic = sum(traffic_detail.values()) / len(traffic_detail)
        except Exception:
            traffic = None

    def roof(prefix, label):
        sel = {k: v for k, v in timer.items() if k.startswith(prefix)}
        if not sel:
            return None
        tot_ms = sum(v[0] for v in sel.values())
        tot_fl = sum(v[2] for v in sel.values())
        n_l = sum(v[1] for v in sel.values())
        ach = tot_fl / (tot_ms / 1e3) / 1e12
        return {"kernel": label % (n_l // max(args.steps, 1)), "bound": "tensor", "achieved": ach, "peak": pk["tflops"],
                "unit": "TFLOP/s", "frac": ach / pk["tflops"],
                "peak_source": pk["source"] + " bf16 sustained (kernels timed inside a long step)",
                "share_of_step": tot_ms / ms_timed, "avg_launch_ms": tot_ms / max(n_l, 1),
                "algorithmic_gflop_per_step": tot_fl / 1e9 / args.steps,
                "per_class": {k: {"ms_per_launch": round(v[0] / v[1], 4), "launches_per_step": v[1] // args.steps,
                                  "tflops": round(v[2] / (v[0] / 1e3) / 1e12, 1)} for k, v in sel.items()}}

    roofline = roof("attn:", "um_window_attention_planes (fused QK^T.softmax.V on tcgen05, %d launches/step)")
    if roofline:
        roofline["traffic"] = traffic
        roofline["traffic_unit"] = "bytes/launch (dram read+write, mean over the launch classes; profiles/r02_ncu_kernels.md)"
        roofline["traffic_per_class"] = traffic_detail
        roofline["ceiling_note"] = "fp32-faithful products need 3 fp16 MMAs each: the path's tensor ceiling is peak/3 (frac 0.333)"
    roofline_conv = roof("conv", "um_conv2d_tc + um_ffn_tc (implicit-GEMM convolutions, Linear layers and the fused FFN on tcgen05, %d launches/step)")
    roofline_simt = roof("attn_simt:", "um_window_attention (CUDA-core kernel: 1-D / small windows, %d launches/step)")

    result = {"metric": metric, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
              "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
              "vs_baseline": None, "dtype": "fp32", "arithmetic": ARITHMETIC, "data": "synthetic", "config": config, "clocks": clocks,
              "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": int(sum(pinned[k].numel() * 4 for k in ("img0", "img1"))),
                      "d2h_bytes_per_step": int(out_host.numel() * 4)},
              "gpu_launches": launches, "cuda_graph": bool(use_graph), "ms_per_step_with_kernel_timers": ms_timed / args.steps,
              "roofline": roofline, "roofline_conv": roofline_conv, "roofline_attention_simt": roofline_simt,
              "sections_ms_per_step": {k[4:]: round(v[0] / args.steps, 3) for k, v in timer.items() if k.startswith("sec:")},
              "ranks": rank_stats, "gather_only_ms": gather_ms}
    if dumped:
        result["dump_outputs"] = dumped

    parity_ok = True
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        one = {k: v[:1] for k, v in host.items()}
        ref, sec = run_oracle_once(sd, cfg, one, ncores)
        mean, mx = error_vs(ref, flow[:1].cpu())
        parity_ok = bool(mean <= tol_mean and mx <= tol_max)
        result["cpu_baseline"] = {"value": 1.0 / sec, "unit": "pairs/s", "cores": ncores, "host_logical_cpus": os.cpu_count(), "kind": "port",
                                  "sample": "1 pair (%dx%d), single run of the oracle port on all physical cores, %.1f s" % (H, W, sec)}
        result["epe_vs_reference"] = {"mean": mean, "max": max(mx, 0.0), "unit": err_unit, "tolerance_mean": tol_mean,
                                      "tolerance_max": tol_max, "pass": parity_ok,
                                      "reference_self_noise": "2e-5 px mean / 1.3e-4 px max under a 1e-7 relative input perturbation (tools/self_noise.py --bench-set)",
                                      "note": "GPU output vs CPU oracle (== reference bit-for-bit, tests/golden) on pair 0 of this batch"}
        if not args.no_ref_gpu:
            # like-for-like GPU baseline (SURVEY.md section 8d): the reference's eager op sequence on this B200, fp32, TF32 off
            try:
                torch.backends.cuda.matmul.allow_tf32 = False
                torch.backends.cudnn.allow_tf32 = False
                nb = min(Bp, 2)
                small = {k: v[:nb] for k, v in host.items()}
                run_oracle_once(sd, cfg, small, ncores, device=dev)
                ts = [run_oracle_once(sd, cfg, small, ncores, device=dev)[1] for _ in range(2)]
                result["reference_eager_gpu"] = {"value": nb / min(ts), "unit": "pairs/s", "batch": nb, "tf32": False,
                                                 "kind": "oracle port (the reference's ATen op sequence) on cuda:%d, eager, best of 2" % local_rank}
            except Exception as e:                          # e.g. out of memory at this batch: report, do not fail the bench
                result["reference_eager_gpu"] = {"error": repr(e)[:200]}
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()
    if not parity_ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
