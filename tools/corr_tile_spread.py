"""Spread of the integer tap origins inside the pixel tiles of the tensor-core correlation volume (um_local_tc.cu), on the
bench's own inputs: runs the CPU oracle forward of gmflow-scale2-regrefine6 (synthetic weights seed 326, one 480x832 pair)
and reports, for every refinement call, the per-tile spread of floor(x + u) - x and floor(y + v) - y, the bounding box of the
tile's 10 x 10 windows and the number of 32 x 8 chunks the kernel needs (more than 6: the tile takes the CUDA-core path).
The tensor-core kernel only pays while the flow is this smooth; rerun when the weights or the inputs change.

    python tools/corr_tile_spread.py [pair index]          (CPU only, about a minute per pair)
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import unimatch_oracle as O  # noqa: E402
from unimatch_b200.spec import WORKLOADS  # noqa: E402
from unimatch_b200.synthetic import BENCH_WEIGHTS, synthetic_batch, synthetic_state_dict  # noqa: E402

TH, TW, CSTEP, MAX_CHUNKS = 8, 16, 23, 6          # um_local_tc.cu


def main():
    cfg = WORKLOADS["gmflow-scale2-regrefine6"]
    sd = synthetic_state_dict(seed=326, **BENCH_WEIGHTS, **cfg["model"])
    orig = O.local_corr_volume

    def hook(f0, f1, flow, radius):
        b, _, h, w = f0.shape
        u, v = flow[:, 0], flow[:, 1]
        ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
        X0, Y0 = torch.floor(xs + u), torch.floor(ys + v)
        hh, ww = (h // TH) * TH, (w // TW) * TW

        def spread(Z, off):
            Zt = (Z[:, :hh, :ww] - off[:hh, :ww]).reshape(b, hh // TH, TH, ww // TW, TW)
            return Zt.amax((2, 4)) - Zt.amin((2, 4))

        sx, sy = spread(X0, xs), spread(Y0, ys)
        zero = torch.zeros_like(xs)
        ax, ay = spread(X0, zero), spread(Y0, zero)          # spread of the absolute tap origins: what the kernel boxes
        chunks = (torch.div(ax, CSTEP, rounding_mode="floor") + 1) * torch.div(ay + 10 + 7, 8, rounding_mode="floor")
        q = lambda t: [round(t.float().quantile(p).item(), 1) for p in (0.5, 0.9, 0.99, 1.0)]
        print(dict(h=h, w=w, tile=(TH, TW), mean_abs_flow=round(flow.abs().mean().item(), 3),
                   spread_x_p50_p90_p99_max=q(sx), spread_y_p50_p90_p99_max=q(sy),
                   box_cols=q(ax + 10), box_rows=q(ay + 10), chunks=q(chunks),
                   frac_tiles_on_tensor_cores=round((chunks <= MAX_CHUNKS).float().mean().item(), 4)), flush=True)
        return orig(f0, f1, flow, radius)

    O.local_corr_volume = hook
    idx = int(sys.argv[1]) if len(sys.argv) > 1 else 0
    batch = synthetic_batch("flow", 1, 480, 832, first_index=idx)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    mk = {k: cfg["model"][k] for k in ("num_scales", "upsample_factor", "reg_refine")}
    t = time.time()
    O.forward(sd, batch["img0"], batch["img1"], **mk, **cfg["call"])
    print("done in %.0f s" % (time.time() - t))


if __name__ == "__main__":
    main()
