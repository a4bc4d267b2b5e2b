"""CUDA-event timing of the refinement's correlation volume on the inputs of a bench forward (gmflow-scale2-regrefine6,
8 pairs at 480x832 -> 8 x 120 x 208 features): the tensor-core op (um_local_corr_volume_planes, volume written into the
update block's operand planes) against the fp32 gather kernel (um_local_corr_volume) followed by the split into those planes,
alternating, for each of the 6 refinement flows.  Reports the fallback tiles, the algorithmic bytes and dot-product FLOPs
and the achieved rates against the B200 data-sheet peaks.

    python tools/profile_local_corr.py [--reps 50] [--pairs 8]
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from unimatch_b200 import UniMatch  # noqa: E402
from unimatch_b200.spec import WORKLOADS  # noqa: E402
from unimatch_b200.synthetic import BENCH_WEIGHTS, synthetic_batch, synthetic_state_dict  # noqa: E402

OPS = torch.ops.unimatch_sm100
HBM_PEAK = 7.7e12              # B/s, HGX B200 data sheet, one GPU
FP16_PEAK = 2.25e15            # dense FP16 FLOP/s, same source


def capture(pairs, H=480, W=832):
    cfg = WORKLOADS["gmflow-scale2-regrefine6"]
    sd = synthetic_state_dict(seed=326, **BENCH_WEIGHTS, **cfg["model"])
    model = UniMatch(**cfg["model"]).eval()
    model.load_state_dict(sd, strict=True)
    model = model.cuda()
    batch = {k: v.cuda() for k, v in synthetic_batch("flow", pairs, H, W, first_index=0).items()}
    calls = []
    orig = model._stage_refine_iter

    def hook(P, rst, g0, g1, flow, task, want_mask, depth=None):
        calls.append((g0, g1, flow.contiguous().clone()))
        return orig(P, rst, g0, g1, flow, task, want_mask, depth)

    model._stage_refine_iter = hook
    with torch.no_grad():
        model(batch["img0"], batch["img1"], **cfg["call"])
    torch.cuda.synchronize()
    return calls


def timed(fn, reps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--pairs", type=int, default=8)
    a = ap.parse_args()
    calls = capture(a.pairs)
    g0, g1 = calls[0][0], calls[0][1]
    b, h, w, _ = g0.shape
    px = b * h * w
    s0 = torch.empty((2, b, h, w, 128), device="cuda", dtype=torch.float16)
    s1 = torch.empty_like(s0)
    OPS.split_planes(g0, s0, 0)
    OPS.split_planes(g1, s1, 0)
    dst = torch.zeros((2, b, h, w, 128), device="cuda", dtype=torch.float16)
    cnt = torch.zeros((1,), device="cuda", dtype=torch.int32)
    tiles = b * ((h + 7) // 8) * ((w + 15) // 16)
    nbytes = px * (512 + 512 + 8 + 81 * 4)      # f0, f1 planes read once, flow, (hi, lo) volume written once
    flops = px * 100 * 128 * 2                  # the 10 x 10 integer-tap dots of 128 channels
    print("device %s | %d x %d x %d features | %d tiles/call | algorithmic %.1f MB, %.2f GFLOP (dots) per call"
          % (torch.cuda.get_device_name(), b, h, w, tiles, nbytes / 1e6, flops / 1e9))
    print("| call | fallback tiles | tensor-core op ms | fp32 gather + split ms | speed-up | GB/s (share of 7.7 TB/s) | "
          "dot TFLOP/s (share of 2250) |\n|---|---|---|---|---|---|---|")
    tot_new = tot_old = 0.0
    for i, (_, _, flow) in enumerate(calls):
        new = lambda: OPS.local_corr_volume_planes(s0, s1, flow, h, w, 4, None, dst, 0, None)
        old = lambda: OPS.split_planes(OPS.local_corr_volume(g0, g1, flow, h, w, 4), dst, 0)
        for f in (new, old, new, old):
            f()
        OPS.local_corr_volume_planes(s0, s1, flow, h, w, 4, None, dst, 0, cnt)
        ms_new, ms_old = [], []
        for _ in range(3):                      # alternate the two paths
            ms_new.append(timed(new, a.reps))
            ms_old.append(timed(old, a.reps))
        tn, to = min(ms_new), min(ms_old)
        tot_new += tn
        tot_old += to
        print("| %d | %d | %.4f | %.4f | %.2fx | %.0f (%.3f) | %.1f (%.4f) |"
              % (i, int(cnt.item()), tn, to, to / tn, nbytes / tn / 1e6, nbytes / tn / 1e-3 / HBM_PEAK,
                 flops / tn / 1e9, flops / tn / 1e-3 / FP16_PEAK), flush=True)
    print("total over the %d calls: tensor-core %.3f ms, fp32 gather + split %.3f ms" % (len(calls), tot_new, tot_old))


if __name__ == "__main__":
    main()
