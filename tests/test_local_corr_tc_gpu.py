"""The tensor-core correlation volume (um_local_corr_volume_planes) against the CPU reference at small shapes and against the
fp32 gather kernel (um_local_corr_volume) at the refinement's own shape, on its tensor-core path, on its CUDA-core path for
rough flows, and with both in one batch.  Tolerances as in test_ops_gpu.py: max |diff| <= TOL * max(1, max |ref|)."""
import ctypes

import pytest
import torch

import refops
from unimatch_b200 import ops

OPS = torch.ops.unimatch_sm100
C = 128
gpu = pytest.mark.gpu


def g(seed):
    return torch.Generator().manual_seed(seed)


def close(got, ref, tol):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    assert torch.isfinite(got).all()
    err = (got - ref).abs().max().item()
    lim = tol * max(1.0, ref.abs().max().item())
    assert err <= lim, "max|diff| %.3e > %.3e" % (err, lim)


def planes(x):
    """fp32 [B, h, w, 128] (CUDA) -> fp16 (hi, lo) planes [2, B, h, w, 128]."""
    p = torch.empty((2,) + tuple(x.shape), device=x.device, dtype=torch.float16)
    OPS.split_planes(x, p, 0)
    return p


def volume(f0, f1, flow, h, w):
    """(fp32 volume, fallback tile count) of the tensor-core op on CUDA inputs."""
    out = torch.empty(f0.shape[:3] + (81,), device=f0.device)
    cnt = torch.full((1,), -1, device=f0.device, dtype=torch.int32)
    OPS.local_corr_volume_planes(planes(f0), planes(f1), flow, h, w, 4, out, None, 0, cnt)
    return out, int(cnt.item())


def smooth_flow(gen, b, h, w, mag, ctrl=(4, 7)):
    """A smooth field like a real flow: bilinear interpolation of a coarse random grid."""
    c = torch.randn((b, 2, *ctrl), generator=gen) * mag
    return torch.nn.functional.interpolate(c, size=(h, w), mode="bilinear", align_corners=True).permute(0, 2, 3, 1).contiguous()


@gpu
@pytest.mark.parametrize("b,h,w,fd,kind,mag", [
    (2, 11, 13, 2, "noise", 3.0),       # one partial tile per image, windows over every border
    (1, 20, 33, 2, "noise", 12.0),      # rough: CUDA-core tiles
    (2, 9, 17, 1, "noise", 4.0),        # disparity
    (1, 8, 8, 2, "noise", 0.0),
    (3, 37, 70, 2, "smooth", 6.0),      # tensor-core tiles, h and w not multiples of the 8 x 16 tile
    (2, 24, 48, 1, "smooth", 5.0),      # disparity, tensor-core tiles
    (1, 19, 35, 2, "const", 25.0),      # every window entirely outside the image
])
def test_local_corr_volume_planes_vs_reference(b, h, w, fd, kind, mag):
    gen = g(4100 + h * w + fd)
    f0 = torch.randn((b, h, w, C), generator=gen)
    f1 = torch.randn((b, h, w, C), generator=gen)
    if kind == "noise":
        flow = torch.randn((b, h, w, fd), generator=gen) * mag
    elif kind == "smooth":
        flow = smooth_flow(gen, b, h, w, mag, (3, 4))[..., :fd].contiguous()
    else:
        flow = torch.full((b, h, w, fd), mag)
    ref = refops.local_corr_volume(f0, f1, flow, h, w, 4)
    got, _ = volume(f0.cuda(), f1.cuda(), flow.cuda(), h, w)
    close(got, ref, 3e-5)


FULL = (8, 120, 208)


def full_inputs(seed):
    b, h, w = FULL
    gen = g(seed)
    f0 = torch.randn((b, h, w, C), generator=gen).cuda()
    f1 = torch.randn((b, h, w, C), generator=gen).cuda()
    return gen, f0, f1


@gpu
def test_smooth_flow_runs_on_tensor_cores_at_refinement_shape():
    b, h, w = FULL
    gen, f0, f1 = full_inputs(4200)
    flow = smooth_flow(gen, b, h, w, 6.0).cuda()
    got, fallback = volume(f0, f1, flow, h, w)
    assert fallback == 0
    close(got, OPS.local_corr_volume(f0, f1, flow, h, w, 4), 3e-5)


@gpu
def test_noise_flow_takes_the_cuda_core_path_at_refinement_shape():
    b, h, w = FULL
    gen, f0, f1 = full_inputs(4300)
    flow = (torch.randn((b, h, w, 2), generator=gen) * 30).cuda()
    got, fallback = volume(f0, f1, flow, h, w)
    assert fallback > 0
    close(got, OPS.local_corr_volume(f0, f1, flow, h, w, 4), 3e-5)


@gpu
def test_mixed_batch_at_refinement_shape():
    b, h, w = FULL
    gen, f0, f1 = full_inputs(4400)
    flow = smooth_flow(gen, b, h, w, 6.0)
    flow[b // 2:] = torch.randn((b - b // 2, h, w, 2), generator=gen) * 30
    flow = flow.cuda()
    got, fallback = volume(f0, f1, flow, h, w)
    tiles = b * ((h + 7) // 8) * ((w + 15) // 16)
    assert 0 < fallback < tiles
    close(got, OPS.local_corr_volume(f0, f1, flow, h, w, 4), 3e-5)


@gpu
def test_zero_flow_equals_shifted_dots_fullsize():
    b, h, w = 1, 120, 208
    gen = g(4500)
    d0 = torch.randn((b, h, w, C), generator=gen).cuda()
    d1 = torch.randn((b, h, w, C), generator=gen).cuda()
    got, fallback = volume(d0, d1, torch.zeros(b, h, w, 2).cuda(), h, w)
    assert fallback == 0
    pad = torch.nn.functional.pad(d1, (0, 0, 4, 4, 4, 4))
    for k in (0, 8, 40, 44, 80):
        iy, ix = k // 9, k % 9
        ref = (d0 * pad[:, iy:iy + h, ix:ix + w]).sum(-1) / (C ** 0.5)
        assert (got[..., k] - ref).abs().max().item() <= 1e-4


@gpu
@pytest.mark.parametrize("off,kind", [(0, "smooth"), (24, "smooth"), (0, "noise")])
def test_planes_output_is_the_split_of_the_fp32_output(off, kind):
    b, h, w = 2, 40, 72
    gen = g(4600 + off)
    f0 = torch.randn((b, h, w, C), generator=gen).cuda()
    f1 = torch.randn((b, h, w, C), generator=gen).cuda()
    flow = (smooth_flow(gen, b, h, w, 5.0, (3, 4)) if kind == "smooth" else torch.randn((b, h, w, 2), generator=gen) * 20).cuda()
    sentinel = torch.randn((2, b, h, w, 128), generator=gen).half().cuda()
    dst = sentinel.clone()
    out = torch.empty((b, h, w, 81), device="cuda")
    OPS.local_corr_volume_planes(planes(f0), planes(f1), flow, h, w, 4, out, dst, off, None)
    want = torch.zeros((2, b, h, w, 81), device="cuda", dtype=torch.float16)
    OPS.split_planes(out, want, 0)
    assert torch.equal(dst[..., off:off + 81], want)
    assert torch.equal(dst[..., :off], sentinel[..., :off])
    assert torch.equal(dst[..., off + 81:], sentinel[..., off + 81:])
    only = sentinel.clone()
    OPS.local_corr_volume_planes(planes(f0), planes(f1), flow, h, w, 4, None, only, off, None)
    assert torch.equal(only, dst)


def test_planes_entry_validates_arguments_without_a_gpu():
    """um_local_corr_volume_planes rejects malformed arguments with -EINVAL and a message before touching the device."""
    one = 1024                                     # any non-null, 16-byte aligned address: validation never dereferences it
    ok = dict(f0=one, f1=one, flow=one, corr=one, split=None, cp=0, off=0, b=1, h=16, w=16, r=4, fd=2)
    bad = [dict(f0=None), dict(flow=None), dict(b=0), dict(h=1), dict(r=3), dict(fd=3), dict(corr=None),
           dict(f1=one + 8), dict(split=one, cp=100, off=24), dict(split=one, cp=128, off=-1)]
    for change in bad:
        a = dict(ok, **change)
        vp = lambda x: ctypes.c_void_p(x) if x is not None else None
        rc = ops.LIB.um_local_corr_volume_planes(vp(a["f0"]), vp(a["f1"]), vp(a["flow"]), vp(a["corr"]), vp(a["split"]),
                                                 a["cp"], a["off"], a["b"], a["h"], a["w"], a["r"], a["fd"], None, None)
        assert rc == -22, change
        assert b"um_local_corr_volume_planes" in ops.LIB.um_last_error(), change
