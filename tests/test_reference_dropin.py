"""Drop-in check against the reference's own flow inference entry point.  tests/golden/golden_dropin.pt holds three small
demo frames and the flows that the reference's unmodified `main_flow.main()` wrote for them (`--inference_size 256 448`,
the synthetic gmflow-scale1 checkpoint below loaded through `--resume --strict_resume`; tests/golden/make_golden_dropin.py).
Here `unimatch_b200.UniMatch` is built with the entry point's constructor arguments, loads the same checkpoint file the
same way (`checkpoint['model']`, strict) and runs through `unimatch_b200.infer_flow` (resize to the inference size,
forward, resize back and rescale): on the CPU kernels of tests/refops.py, and on cuda:0 with the CUDA kernels."""
import os

import pytest
import torch

from unimatch_b200.spec import WORKLOADS
from unimatch_b200.synthetic import BENCH_WEIGHTS, synthetic_state_dict

GOLD = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_dropin.pt"))


def check_against_reference_entry_point(device, tmp_path):
    import unimatch_b200
    wl = WORKLOADS["gmflow-scale1"]
    ckpt = str(tmp_path / "synthetic.pth")
    torch.save({"model": synthetic_state_dict(seed=326, **BENCH_WEIGHTS, **wl["model"])}, ckpt)
    model = unimatch_b200.UniMatch(feature_channels=128, num_scales=1, upsample_factor=8, num_head=1, ffn_dim_expansion=4,
                                   num_transformer_layers=6, reg_refine=False, task="flow")
    model.load_state_dict(torch.load(ckpt, map_location="cpu")["model"], strict=True)
    model = model.to(device).eval()
    frames = GOLD["frames"].permute(0, 3, 1, 2).float().to(device)          # uint8 [N, H, W, 3] -> [N, 3, H, W] in [0, 255]
    call = {k: v for k, v in wl["call"].items() if k != "task"}
    flow = unimatch_b200.infer_flow(model, frames[:-1], frames[1:], padding_factor=16,
                                    inference_size=GOLD["inference_size"], **call)["flow"]
    n = len(GOLD["files"])
    assert n >= 2 and flow.shape == (n, 2) + tuple(frames.shape[-2:]) and flow.dtype == torch.float32
    got = flow.permute(0, 2, 3, 1).reshape(n, -1, 2)[:, GOLD["pixels"].to(device)].cpu()
    epe = (got - GOLD["flows"]).norm(dim=-1)
    # same weights, same frames, fp32 both sides: the flows agree to ~1e-5 px on the CPU kernels; stated tolerance 1e-2 px
    # mean as everywhere (tests/stage_checks.py)
    assert epe.mean().item() <= 1e-2 and epe.max().item() <= 1e-1, (epe.mean().item(), epe.max().item())


def test_dropin_class_reproduces_the_reference_flow_entry_point(tmp_path):
    import refops
    refops.register_cpu_kernels()
    check_against_reference_entry_point("cpu", tmp_path)


@pytest.mark.gpu
def test_dropin_class_reproduces_the_reference_flow_entry_point_on_gpu(tmp_path):
    check_against_reference_entry_point("cuda", tmp_path)
