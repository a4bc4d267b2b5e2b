"""Generate tests/golden/golden_dropin.pt by running the REFERENCE's unmodified flow inference entry point.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_dropin.py REFERENCE_CHECKOUT

Takes the first three frames of the reference's `demo/flow-davis`, shrinks them 8x (box filter) to 60x107 uint8 frames,
writes them as PNG (lossless) and runs the reference's `main_flow.main()` on them (`--inference_size 256 448`, the same
synthetic gmflow-scale1 checkpoint that `tests/test_reference_dropin.py` builds, loaded through `--resume --strict_resume`).
Stores the frames, and the `.flo` flows the reference writes at a fixed seeded sample of pixels, for that test.
`imageio`, `skimage(.io)` and `matplotlib(.cm)` are import-time-only dependencies of the reference's drivers; they are
stubbed when missing.
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
FRAME_HW = (60, 107)
SAMPLES = 1024
ARGV = ["--inference_size", "256", "448", "--padding_factor", "16", "--upsample_factor", "8", "--num_scales", "1",
        "--attn_splits_list", "2", "--corr_radius_list", "-1", "--prop_radius_list", "-1"]


def stub_driver_imports():
    for name in ("imageio", "skimage", "skimage.io", "matplotlib", "matplotlib.cm", "matplotlib.pyplot"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    if not hasattr(sys.modules["skimage"], "io"):
        sys.modules["skimage"].io = sys.modules["skimage.io"]
    if not hasattr(sys.modules["matplotlib"], "cm"):
        sys.modules["matplotlib"].cm = sys.modules["matplotlib.cm"]
    if not hasattr(sys.modules["matplotlib.cm"], "get_cmap"):
        sys.modules["matplotlib.cm"].get_cmap = lambda *a, **k: None


def read_flo(path):
    with open(path, "rb") as f:
        assert np.fromfile(f, np.float32, 1)[0] == 202021.25
        w, h = np.fromfile(f, np.int32, 2)
        return np.fromfile(f, np.float32, 2 * w * h).reshape(h, w, 2)


def main():
    ref = os.path.abspath(sys.argv[1])
    sys.dont_write_bytecode = True
    sys.path[:0] = [ref, ROOT]
    stub_driver_imports()
    import main_flow                                     # the reference entry script, unmodified
    from unimatch_b200.spec import WORKLOADS
    from unimatch_b200.synthetic import BENCH_WEIGHTS, synthetic_state_dict

    demo = os.path.join(ref, "demo", "flow-davis")
    names = sorted(f for f in os.listdir(demo) if f.endswith(".jpg"))[:3]
    frames = np.stack([np.asarray(Image.open(os.path.join(demo, n)).convert("RGB").resize(FRAME_HW[::-1], Image.BOX))
                       for n in names])
    torch.set_num_threads(8)
    with tempfile.TemporaryDirectory() as tmp:
        src, out = os.path.join(tmp, "frames"), os.path.join(tmp, "flow")
        os.makedirs(src)
        for i, fr in enumerate(frames):
            Image.fromarray(fr).save(os.path.join(src, "%05d.png" % i))
        ckpt = os.path.join(tmp, "synthetic.pth")
        torch.save({"model": synthetic_state_dict(seed=326, **BENCH_WEIGHTS, **WORKLOADS["gmflow-scale1"]["model"])}, ckpt)
        argv = ["--inference_dir", src, "--output_path", out, "--resume", ckpt, "--strict_resume", "--save_flo_flow"] + ARGV
        main_flow.main(main_flow.get_args_parser().parse_args(argv))
        flo = sorted(f for f in os.listdir(out) if f.endswith(".flo"))
        flows = np.stack([read_flo(os.path.join(out, f)) for f in flo])
    assert flows.shape == (len(frames) - 1,) + FRAME_HW + (2,), flows.shape
    idx = torch.randperm(FRAME_HW[0] * FRAME_HW[1], generator=torch.Generator().manual_seed(0))[:SAMPLES].sort().values
    golden = {"frames": torch.from_numpy(frames), "pixels": idx,
              "flows": torch.from_numpy(flows).reshape(len(flo), -1, 2)[:, idx].contiguous(), "files": flo,
              "inference_size": (256, 448)}
    path = os.path.join(HERE, "golden_dropin.pt")
    torch.save(golden, path)
    print("wrote %s (%.1f kB): frames %s, flows %s, mean |flow| %.3f px" % (
        path, os.path.getsize(path) / 1e3, tuple(frames.shape), tuple(golden["flows"].shape),
        float(np.linalg.norm(flows, axis=-1).mean())))


if __name__ == "__main__":
    main()
