"""ctypes binding of libunimatch_sm100.so + registration of every entry point as a torch custom op
(`torch.ops.unimatch_sm100.*`, CUDA only).

There is no CPU or PyTorch fallback on this path: if the shared library is missing it is built with nvcc,
and if that is impossible the import fails; an op called with CPU tensors raises (no CPU kernel is registered).
The C ABI is declared in include/unimatch_sm100.h.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libunimatch_sm100.so")

# every symbol include/unimatch_sm100.h declares (checked by tests/test_cabi.py)
SYMBOLS = [
    "um_abi_version", "um_build_info", "um_last_error", "um_launch_count",
    "um_window_attention", "um_window_attention_workspace", "um_attention_planes_lp", "um_window_attention_planes", "um_debug_set_dump", "um_softmax_expectation", "um_softmax_expectation_workspace",
    "um_local_corr_softmax", "um_local_corr_volume", "um_local_corr_volume_planes", "um_flow_warp", "um_fb_consistency", "um_propagate_local", "um_depth_corr_softmax",
    "um_conv2d_tc", "um_ffn_tc", "um_conv7x7_small", "um_split_planes", "um_instance_norm_scratch_floats", "um_instance_norm_stats", "um_instance_norm_apply", "um_add_position", "um_layernorm_residual", "um_convex_upsample", "um_upsample2x", "um_resize_bilinear", "um_gru_rh", "um_gru_update",
]

MASK_NONE, MASK_SWIN, MASK_CAUSAL = 0, 1, 2
VALUE_TENSOR, VALUE_COORDS, VALUE_XCOORD = 0, 1, 2
POST_NONE, POST_MINUS_OWN, POST_OWN_MINUS = 0, 1, 2


FORCE_CUDA_CORES = 1
_force_cuda_cores = False      # diagnostic switch (tests): route every attention shape to the exact-fp32 CUDA-core kernel


def set_force_cuda_cores(flag):
    global _force_cuda_cores
    _force_cuda_cores = bool(flag)


ACT_NONE, ACT_RELU, ACT_TANH, ACT_SIGMOID, ACT_GELU = 0, 1, 2, 3, 4
CONV_LINEAR, CONV_GRU_ZR, CONV_GRU_Q, CONV_LN = 0, 1, 2, 3


class AttnGeom(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("h", "w", "kh", "kw", "sh", "sw", "mask_mode")]


class ConvDesc(ctypes.Structure):
    _fields_ = [("src", ctypes.c_void_p * 2), ("cin_p", ctypes.c_int32 * 2), ("nsrc", ctypes.c_int32),
                ("batch", ctypes.c_int32), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
                ("weights", ctypes.c_void_p), ("bias", ctypes.c_void_p),
                ("kh", ctypes.c_int32), ("kw", ctypes.c_int32), ("pad_h", ctypes.c_int32), ("pad_w", ctypes.c_int32),
                ("cout", ctypes.c_int32), ("cout_p", ctypes.c_int32), ("bn", ctypes.c_int32),
                ("mode", ctypes.c_int32), ("act", ctypes.c_int32),
                ("out_f32", ctypes.c_void_p), ("ld_f32", ctypes.c_int64), ("off_f32", ctypes.c_int32),
                ("cp_split", ctypes.c_int32), ("out_split", ctypes.c_void_p), ("off_split", ctypes.c_int32),
                ("stride", ctypes.c_int32),
                ("aux0", ctypes.c_void_p), ("ld_aux0", ctypes.c_int64), ("aux1", ctypes.c_void_p), ("ld_aux1", ctypes.c_int64),
                ("gamma", ctypes.c_void_p), ("beta", ctypes.c_void_p),
                ("src_plane_stride", ctypes.c_int64), ("split_plane_stride", ctypes.c_int64),
                ("win_dst", ctypes.c_void_p), ("win_c0", ctypes.c_int32), ("win_c1", ctypes.c_int32),
                ("win_lp", ctypes.c_int32), ("win_streams", ctypes.c_int32), ("win_geom", AttnGeom),
                ("pre", ctypes.c_void_p), ("ld_pre", ctypes.c_int64)]


class FfnDesc(ctypes.Structure):
    _fields_ = [("src", ctypes.c_void_p * 2), ("src_plane_stride", ctypes.c_int64), ("rows", ctypes.c_int64),
                ("w1", ctypes.c_void_p), ("w2", ctypes.c_void_p), ("hidden", ctypes.c_int32),
                ("residual", ctypes.c_void_p), ("ld_res", ctypes.c_int64), ("gamma", ctypes.c_void_p), ("beta", ctypes.c_void_p),
                ("out_f32", ctypes.c_void_p), ("ld_f32", ctypes.c_int64), ("out_split", ctypes.c_void_p),
                ("split_plane_stride", ctypes.c_int64)]


def _load():
    from .csrc.build import build, have_nvcc
    if have_nvcc():
        build()                         # no-op when the in-tree .so matches the sources (content stamp)
    elif not os.path.exists(LIB_PATH):  # no library and no compiler: the product path has no fallback
        raise ImportError("libunimatch_sm100.so is missing and nvcc is not available to build it")
    lib = ctypes.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise ImportError("libunimatch_sm100.so lacks symbols %s (stale build? run python unimatch_b200/csrc/build.py --force)" % missing)
    lib.um_build_info.restype = ctypes.c_char_p
    lib.um_last_error.restype = ctypes.c_char_p
    lib.um_launch_count.restype = ctypes.c_int64
    P, I, L, F = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
    G = ctypes.POINTER(AttnGeom)
    sig = {
        "um_window_attention": [P, P, P, P, I, I, L, L, L, L, G, P, L, I, P],
        "um_softmax_expectation": [P, P, P, P, I, I, I, L, L, I, I, I, G, P, L, I, P],
        "um_local_corr_softmax": [P, P, P, I, I, I, I, I, I, P],
        "um_local_corr_volume": [P, P, P, P, I, I, I, I, I, P],
        "um_local_corr_volume_planes": [P, P, P, P, P, I, I, I, I, I, I, I, P, P],
        "um_flow_warp": [P, P, P, I, I, I, I, P],
        "um_fb_consistency": [P, P, F, F, P, P, I, I, I, P],
        "um_propagate_local": [P, P, P, P, I, I, I, I, I, L, L, P],
        "um_depth_corr_softmax": [P, P, P, P, P, P, P, I, I, I, I, I, P],
        "um_add_position": [P, P, P, I, I, I, I, I, P],
        "um_layernorm_residual": [P, P, P, P, P, L, L, L, L, P],
        "um_convex_upsample": [P, P, P, I, I, I, I, I, F, P],
        "um_upsample2x": [P, P, I, I, I, I, F, P],
        "um_gru_rh": [P, L, P, L, P, L, L, P],
        "um_gru_update": [P, L, P, L, P, L, P, L, L, P],
    }
    lib.um_window_attention_workspace.argtypes = [G, I]
    lib.um_window_attention_workspace.restype = ctypes.c_int64
    lib.um_softmax_expectation_workspace.argtypes = [G, I, I]
    lib.um_softmax_expectation_workspace.restype = ctypes.c_int64
    lib.um_conv2d_tc.argtypes = [ctypes.POINTER(ConvDesc), P]
    lib.um_conv2d_tc.restype = ctypes.c_int
    lib.um_ffn_tc.argtypes = [ctypes.POINTER(FfnDesc), P]
    lib.um_ffn_tc.restype = ctypes.c_int
    lib.um_split_planes.argtypes = [P, L, I, L, P, I, I, L, P]
    lib.um_attention_planes_lp.argtypes = [G]
    lib.um_attention_planes_lp.restype = ctypes.c_int32
    lib.um_window_attention_planes.argtypes = [P, P, P, P, L, P, L, I, I, G, P]
    lib.um_window_attention_planes.restype = ctypes.c_int
    lib.um_split_planes.restype = ctypes.c_int
    FP = ctypes.POINTER(ctypes.c_float)
    lib.um_conv7x7_small.argtypes = [P, P, I, I, I, I, I, I, I, P, P, I, I, FP, FP, P, L, P, I, P]
    lib.um_conv7x7_small.restype = ctypes.c_int
    lib.um_instance_norm_scratch_floats.argtypes = [I, I]
    lib.um_instance_norm_scratch_floats.restype = ctypes.c_int64
    lib.um_instance_norm_stats.argtypes = [P, L, I, I, I, P, P, P]
    lib.um_instance_norm_stats.restype = ctypes.c_int
    lib.um_instance_norm_apply.argtypes = [P, L, P, I, P, L, P, I, P, L, P, I, I, I, I, I, P]
    lib.um_instance_norm_apply.restype = ctypes.c_int
    lib.um_resize_bilinear.argtypes = [P, P, I, I, I, I, I, I, FP, I, P]
    lib.um_resize_bilinear.restype = ctypes.c_int
    lib.um_debug_set_dump.argtypes = [P]
    lib.um_debug_set_dump.restype = None
    for name, argtypes in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    return lib


LIB = _load()


def build_info():
    return LIB.um_build_info().decode()


def launch_count():
    return int(LIB.um_launch_count())


def _check(rc, name):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, LIB.um_last_error().decode()))


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name, rows_ok=False):
    if not t.is_cuda:
        raise RuntimeError("%s: expected a CUDA tensor (libunimatch_sm100 has no CPU path)" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("%s: expected float32" % name)
    if rows_ok:
        if t.stride(-1) != 1:
            raise RuntimeError("%s: last dim must be contiguous" % name)
    elif not t.is_contiguous():
        raise RuntimeError("%s: expected a contiguous tensor" % name)
    return t


def _rows(t, name):
    """[N, L, 128] view with uniform row stride: returns ld (floats)."""
    _f32c(t, name, rows_ok=True)
    if t.dim() != 3 or t.shape[-1] != 128:
        raise RuntimeError("%s: expected [N, L, 128]" % name)
    ld = t.stride(1)
    if t.shape[0] > 1 and t.stride(0) != ld * t.shape[1]:
        raise RuntimeError("%s: batch stride must equal L * row stride" % name)
    return ld


_lib = torch.library.Library("unimatch_sm100", "DEF")


def _define(schema, impl):
    _lib.define(schema)
    name = schema.split("(")[0]
    _lib.impl(name, impl, "CUDA")
    return getattr(torch.ops.unimatch_sm100, name)


# ---- attention ------------------------------------------------------------------------------------------
def _window_attention(q, k, v, kv_shift, h, w, kh, kw, sh, sw, mask_mode):
    ldq, ldk, ldv = _rows(q, "q"), _rows(k, "k"), _rows(v, "v")
    n, l, _ = q.shape
    out = torch.empty((n, l, 128), device=q.device, dtype=torch.float32)
    g = AttnGeom(h, w, kh, kw, sh, sw, mask_mode)
    flags = FORCE_CUDA_CORES if _force_cuda_cores else 0
    ws_bytes = 0 if flags else int(LIB.um_window_attention_workspace(ctypes.byref(g), n))
    ws = torch.empty((ws_bytes,), device=q.device, dtype=torch.uint8) if ws_bytes else None
    _check(LIB.um_window_attention(_p(q), _p(k), _p(v), _p(out), n, kv_shift, ldq, ldk, ldv, 128, ctypes.byref(g),
                                   _p(ws), ws_bytes, flags, _stream()), "um_window_attention")
    return out


window_attention = _define(
    "window_attention(Tensor q, Tensor k, Tensor v, int kv_shift, int h, int w, int kh, int kw, int sh, int sw, "
    "int mask_mode) -> Tensor", _window_attention)


def attention_planes_lp(h, w, kh, kw, sh, sw, mask_mode):
    """Padded window length of the tensor-core attention's operand planes; 0 = this geometry runs on the CUDA-core kernel."""
    g = AttnGeom(h, w, kh, kw, sh, sw, mask_mode)
    return int(LIB.um_attention_planes_lp(ctypes.byref(g)))


def _planes_ok(t, name, n, nwin, lp):
    if t.dtype != torch.float16 or not t.is_contiguous() or t.numel() != 2 * n * nwin * lp * 128:
        raise RuntimeError("%s: expected contiguous fp16 planes [2, %d, %d, %d, 128]" % (name, n, nwin, lp))


def _window_attention_planes(qp, kp, vp, n, kv_shift, h, w, kh, kw, sh, sw, mask_mode, out_f32, out_split):
    g = AttnGeom(h, w, kh, kw, sh, sw, mask_mode)
    lp = int(LIB.um_attention_planes_lp(ctypes.byref(g)))
    if lp == 0:
        raise RuntimeError("window_attention_planes: geometry is not built for the tensor-core kernel")
    for t, nm in ((qp, "q_planes"), (kp, "k_planes"), (vp, "v_planes")):
        _planes_ok(t, nm, n, kh * kw, lp)
    ldo, plane = 0, 0
    if out_f32 is not None:
        ldo = _rows(out_f32, "out_f32")
    if out_split is not None:
        if out_split.dtype != torch.float16 or not out_split.is_contiguous() or out_split.shape[0] != 2 or out_split.shape[-1] != 128:
            raise RuntimeError("window_attention_planes: out_split must be contiguous fp16 planes [2, rows, 128]")
        plane = out_split[0].numel()
    _check(LIB.um_window_attention_planes(_p(qp), _p(kp), _p(vp), _p(out_f32), ldo, _p(out_split), plane, n, kv_shift,
                                          ctypes.byref(g), _stream()), "um_window_attention_planes")


window_attention_planes = _define(
    "window_attention_planes(Tensor q_planes, Tensor k_planes, Tensor v_planes, int n_streams, int kv_shift, int h, int w, "
    "int kh, int kw, int sh, int sw, int mask_mode, Tensor(a!)? out_f32, Tensor(b!)? out_split) -> ()",
    _window_attention_planes)


def _softmax_expectation(q, k, values, n_streams, kv_shift, vdim, value_mode, post_op, h, w, kh, kw, mask_mode):
    ldq, ldk = _rows(q, "q"), _rows(k, "k")
    n_total, l, _ = q.shape
    if values is not None:
        _f32c(values, "values")
    out = torch.empty((n_streams, l, vdim), device=q.device, dtype=torch.float32)
    g = AttnGeom(h, w, kh, kw, 0, 0, mask_mode)
    flags = FORCE_CUDA_CORES if _force_cuda_cores else 0
    ws_bytes = 0 if flags else int(LIB.um_softmax_expectation_workspace(ctypes.byref(g), n_total, value_mode))
    ws = torch.empty((ws_bytes,), device=q.device, dtype=torch.uint8) if ws_bytes else None
    _check(LIB.um_softmax_expectation(_p(q), _p(k), _p(values), _p(out), n_streams, n_total, kv_shift, ldq, ldk, vdim,
                                      value_mode, post_op, ctypes.byref(g), _p(ws), ws_bytes, flags, _stream()),
           "um_softmax_expectation")
    return out


softmax_expectation = _define(
    "softmax_expectation(Tensor q, Tensor k, Tensor? values, int n_streams, int kv_shift, int vdim, int value_mode, "
    "int post_op, int h, int w, int kh, int kw, int mask_mode) -> Tensor", _softmax_expectation)


# ---- local matching ---------------------------------------------------------------------------------------
def _local_corr_softmax(f0, f1, h, w, ry, rx, stereo):
    _f32c(f0, "f0"), _f32c(f1, "f1")
    b = f0.shape[0]
    out = torch.empty((b, h, w, 1 if stereo else 2), device=f0.device, dtype=torch.float32)
    _check(LIB.um_local_corr_softmax(_p(f0), _p(f1), _p(out), b, h, w, ry, rx, int(stereo), _stream()),
           "um_local_corr_softmax")
    return out


local_corr_softmax = _define("local_corr_softmax(Tensor f0, Tensor f1, int h, int w, int ry, int rx, bool stereo) -> Tensor",
                             _local_corr_softmax)


def _local_corr_volume(f0, f1, flow, h, w, radius):
    _f32c(f0, "f0"), _f32c(f1, "f1"), _f32c(flow, "flow")
    b = f0.shape[0]
    k = (2 * radius + 1) ** 2
    out = torch.empty((b, h, w, k), device=f0.device, dtype=torch.float32)
    _check(LIB.um_local_corr_volume(_p(f0), _p(f1), _p(flow), _p(out), b, h, w, radius, flow.shape[-1], _stream()),
           "um_local_corr_volume")
    return out


local_corr_volume = _define("local_corr_volume(Tensor f0, Tensor f1, Tensor flow, int h, int w, int radius) -> Tensor",
                            _local_corr_volume)


def _local_corr_volume_planes(f0_planes, f1_planes, flow, h, w, radius, out_f32, out_split, off_split, fallback_tiles):
    """local_corr_volume on fp16 (hi, lo) feature planes [2, B, h, w, 128] (tensor cores).  Writes out_f32 [B, h, w, 81]
    and/or channels [off_split, off_split + 81) of the planes out_split [2, B, h, w, cp]; fallback_tiles (int32 [1]) receives
    the number of pixel tiles whose flow was too rough for the tensor-core path."""
    b = f0_planes.shape[1]
    for t, name in ((f0_planes, "f0_planes"), (f1_planes, "f1_planes")):
        if t.dtype != torch.float16 or not t.is_contiguous() or tuple(t.shape) != (2, b, h, w, 128):
            raise RuntimeError("local_corr_volume_planes: %s must be contiguous fp16 planes [2, B, h, w, 128]" % name)
    _f32c(flow, "flow")
    if tuple(flow.shape[:3]) != (b, h, w):
        raise RuntimeError("local_corr_volume_planes: flow must be [B, h, w, 1 or 2]")
    k = (2 * radius + 1) ** 2
    if out_f32 is not None:
        _f32c(out_f32, "out_f32")
        if tuple(out_f32.shape) != (b, h, w, k):
            raise RuntimeError("local_corr_volume_planes: out_f32 must be [B, h, w, %d]" % k)
    cp = 0
    if out_split is not None:
        if out_split.dtype != torch.float16 or not out_split.is_contiguous() or tuple(out_split.shape[:4]) != (2, b, h, w):
            raise RuntimeError("local_corr_volume_planes: out_split must be contiguous fp16 planes [2, B, h, w, cp]")
        cp = out_split.shape[-1]
    if fallback_tiles is not None and (fallback_tiles.dtype != torch.int32 or fallback_tiles.numel() < 1):
        raise RuntimeError("local_corr_volume_planes: fallback_tiles must be an int32 tensor")
    _check(LIB.um_local_corr_volume_planes(_p(f0_planes), _p(f1_planes), _p(flow), _p(out_f32), _p(out_split), cp, off_split,
                                           b, h, w, radius, flow.shape[-1], _p(fallback_tiles), _stream()),
           "um_local_corr_volume_planes")


local_corr_volume_planes = _define(
    "local_corr_volume_planes(Tensor f0_planes, Tensor f1_planes, Tensor flow, int h, int w, int radius, Tensor(a!)? out_f32, "
    "Tensor(b!)? out_split, int off_split, Tensor(c!)? fallback_tiles) -> ()", _local_corr_volume_planes)


def _flow_warp(f, flow, h, w):
    _f32c(f, "f"), _f32c(flow, "flow")
    out = torch.empty_like(f)
    _check(LIB.um_flow_warp(_p(f), _p(flow), _p(out), f.shape[0], h, w, flow.shape[-1], _stream()), "um_flow_warp")
    return out


flow_warp = _define("flow_warp(Tensor f, Tensor flow, int h, int w) -> Tensor", _flow_warp)


def _fb_consistency(fwd_flow, bwd_flow, alpha, beta):
    _f32c(fwd_flow, "fwd_flow"), _f32c(bwd_flow, "bwd_flow")
    if fwd_flow.dim() != 4 or fwd_flow.shape[1] != 2 or fwd_flow.shape != bwd_flow.shape:
        raise ValueError("fb_consistency: flows must be planar [B,2,H,W] of equal shape")
    b, _, h, w = fwd_flow.shape
    fwd_occ = torch.empty((b, h, w), device=fwd_flow.device, dtype=torch.float32)
    bwd_occ = torch.empty_like(fwd_occ)
    _check(LIB.um_fb_consistency(_p(fwd_flow), _p(bwd_flow), float(alpha), float(beta), _p(fwd_occ), _p(bwd_occ), b, h, w,
                                 _stream()), "um_fb_consistency")
    return fwd_occ, bwd_occ


fb_consistency = _define("fb_consistency(Tensor fwd_flow, Tensor bwd_flow, float alpha, float beta) -> (Tensor, Tensor)",
                         _fb_consistency)


def _propagate_local(q, k, flow, h, w, radius):
    ldq, ldk = _rows(q, "q"), _rows(k, "k")
    _f32c(flow, "flow")
    b = q.shape[0]
    out = torch.empty_like(flow)
    _check(LIB.um_propagate_local(_p(q), _p(k), _p(flow), _p(out), b, h, w, radius, flow.shape[-1], ldq, ldk, _stream()),
           "um_propagate_local")
    return out


propagate_local = _define("propagate_local(Tensor q, Tensor k, Tensor flow, int h, int w, int radius) -> Tensor",
                          _propagate_local)


def _depth_corr_softmax(f0, f1, K, Kinv, pose, cand, h, w, from_argmax):
    for t, n in ((f0, "f0"), (f1, "f1"), (K, "K"), (Kinv, "Kinv"), (pose, "pose"), (cand, "cand")):
        _f32c(t, n)
    b = f0.shape[0]
    out = torch.empty((b, h, w, 1), device=f0.device, dtype=torch.float32)
    _check(LIB.um_depth_corr_softmax(_p(f0), _p(f1), _p(K), _p(Kinv), _p(pose), _p(cand), _p(out), b, h, w,
                                     cand.numel(), int(from_argmax), _stream()), "um_depth_corr_softmax")
    return out


depth_corr_softmax = _define(
    "depth_corr_softmax(Tensor f0, Tensor f1, Tensor K, Tensor Kinv, Tensor pose, Tensor cand, int h, int w, "
    "bool from_argmax) -> Tensor", _depth_corr_softmax)


# ---- glue -------------------------------------------------------------------------------------------------
def _add_position(x, table, h, w):
    _f32c(x, "x"), _f32c(table, "table")
    out = torch.empty_like(x)
    _check(LIB.um_add_position(_p(x), _p(table), _p(out), x.shape[0], h, w, table.shape[0], table.shape[1], _stream()),
           "um_add_position")
    return out


add_position = _define("add_position(Tensor x, Tensor table, int h, int w) -> Tensor", _add_position)


def _layernorm_residual(x, residual, gamma, beta):
    _f32c(x, "x", rows_ok=True), _f32c(gamma, "gamma"), _f32c(beta, "beta")
    if x.shape[-1] != 128:
        raise RuntimeError("layernorm_residual: expected rows of 128 channels")
    x2 = x.flatten(0, -2)
    rows = x2.shape[0]
    out = torch.empty((rows, 128), device=x.device, dtype=torch.float32)
    ldr, r2 = 0, None
    if residual is not None:
        _f32c(residual, "residual", rows_ok=True)
        r2 = residual.flatten(0, -2)
        ldr = r2.stride(0)
    _check(LIB.um_layernorm_residual(_p(x2), _p(r2), _p(gamma), _p(beta), _p(out), rows, x2.stride(0), ldr, 128,
                                     _stream()), "um_layernorm_residual")
    return out.view(x.shape)


layernorm_residual = _define("layernorm_residual(Tensor x, Tensor? residual, Tensor gamma, Tensor beta) -> Tensor",
                             _layernorm_residual)


def _convex_upsample(flow, mask, factor, mult):
    _f32c(flow, "flow"), _f32c(mask, "mask")
    b, h, w, fd = flow.shape
    out = torch.empty((b, fd, h * factor, w * factor), device=flow.device, dtype=torch.float32)
    _check(LIB.um_convex_upsample(_p(flow), _p(mask), _p(out), b, h, w, fd, factor, float(mult), _stream()),
           "um_convex_upsample")
    return out


convex_upsample = _define("convex_upsample(Tensor flow, Tensor mask, int factor, float mult) -> Tensor", _convex_upsample)


def _upsample2x(flow, mult):
    _f32c(flow, "flow")
    b, h, w, fd = flow.shape
    out = torch.empty((b, 2 * h, 2 * w, fd), device=flow.device, dtype=torch.float32)
    _check(LIB.um_upsample2x(_p(flow), _p(out), b, h, w, fd, float(mult), _stream()), "um_upsample2x")
    return out


upsample2x = _define("upsample2x(Tensor flow, float mult) -> Tensor", _upsample2x)


def _resize_bilinear(x, h_out, w_out, scale, flip_x):
    _f32c(x, "x")
    if x.dim() != 4 or x.shape[1] > 3:
        raise RuntimeError("resize_bilinear: expected planar [B, C <= 3, H, W]")
    b, c, h, w = x.shape
    out = torch.empty((b, c, h_out, w_out), device=x.device, dtype=torch.float32)
    sc = (ctypes.c_float * c)(*scale) if scale is not None else None
    _check(LIB.um_resize_bilinear(_p(x), _p(out), b, c, h, w, h_out, w_out, sc, int(flip_x), _stream()), "um_resize_bilinear")
    return out


resize_bilinear = _define("resize_bilinear(Tensor x, int h_out, int w_out, float[]? scale, bool flip_x) -> Tensor", _resize_bilinear)


def _gru_rh(r_pre, h):
    _f32c(r_pre, "r_pre", rows_ok=True), _f32c(h, "h", rows_ok=True)
    r2, h2 = r_pre.flatten(0, -2), h.flatten(0, -2)
    rows = h2.shape[0]
    out = torch.empty((rows, 128), device=h.device, dtype=torch.float32)
    _check(LIB.um_gru_rh(_p(r2), r2.stride(0), _p(h2), h2.stride(0), _p(out), 128, rows, _stream()), "um_gru_rh")
    return out.view(h.shape)


gru_rh = _define("gru_rh(Tensor r_pre, Tensor h) -> Tensor", _gru_rh)


def _gru_update(z_pre, q_pre, h):
    for t, n in ((z_pre, "z_pre"), (q_pre, "q_pre"), (h, "h")):
        _f32c(t, n, rows_ok=True)
    z2, q2, h2 = z_pre.flatten(0, -2), q_pre.flatten(0, -2), h.flatten(0, -2)
    rows = h2.shape[0]
    out = torch.empty((rows, 128), device=h.device, dtype=torch.float32)
    _check(LIB.um_gru_update(_p(z2), z2.stride(0), _p(q2), q2.stride(0), _p(h2), h2.stride(0), _p(out), 128, rows,
                             _stream()), "um_gru_update")
    return out.view(h.shape)


gru_update = _define("gru_update(Tensor z_pre, Tensor q_pre, Tensor h) -> Tensor", _gru_update)


# ---- tensor-core convolution / Linear ---------------------------------------------------------------------------
def prep_conv_weight(w, cin_splits, cout_p):
    """[Cout, sum(cin_splits), KH, KW] fp32 -> fp16 planes [2, cout_p, ktot], K ordered (source, tap, ci) with every
    source's channels padded to a multiple of 64 (host-side, once per weight)."""
    cout, _, kh, kw = w.shape
    cols, off = [], 0
    for c in cin_splits:
        cp = (c + 63) // 64 * 64
        ws = w[:, off:off + c].permute(0, 2, 3, 1)                      # [Cout, KH, KW, c]
        ws = torch.nn.functional.pad(ws, (0, cp - c)).reshape(cout, kh * kw * cp)
        cols.append(ws)
        off += c
    m = torch.cat(cols, dim=1)
    m = torch.nn.functional.pad(m, (0, 0, 0, cout_p - cout)).float()
    hi = m.half()
    lo = (m - hi.float()).half()
    out = torch.stack((hi, lo), dim=0).contiguous()
    out.k_true = int(w.shape[1] * kh * kw)          # real (unpadded) reduction length: algorithmic FLOPs of the layer
    return out


def split_buffer(batch, h, w, cp, device):
    """Zero-initialised fp16 (hi, lo) activation planes [2, B, h, w, cp]."""
    return torch.zeros((2, batch, h, w, cp), device=device, dtype=torch.float16)


def _split_planes(src, dst, off):
    _f32c(src, "src", rows_ok=True)
    s2 = src.flatten(0, -2)
    rows, c = s2.shape
    cp = dst.shape[-1]
    if dst.dtype != torch.float16 or not dst.is_contiguous() or dst.shape[0] != 2 or dst[0].numel() < rows * cp:
        raise RuntimeError("split_planes: dst must be contiguous fp16 planes [2, >= rows, cp]")
    _check(LIB.um_split_planes(_p(s2), rows, c, s2.stride(0), _p(dst), cp, off, dst[0].numel(), _stream()), "um_split_planes")


split_planes = _define("split_planes(Tensor src, Tensor(a!) dst, int off) -> ()", _split_planes)


def _conv2d_tc(src0, src1, weights, bias, kh, kw, pad_h, pad_w, cout, bn, mode, act, out_f32, off_f32, out_split,
               off_split, aux0, aux1, gamma=None, beta=None, stride=1, rows=0, win_dst=None, win_geom=None, win_c0=0,
               win_c1=0, win_streams=0, pre=None):
    """`rows` > 0: the sources / out_split are [2, R, cp] plane buffers of token rows and the layer runs over their first
    `rows` rows as a [rows/16, 16] pixel grid (rows % 16 == 0), the (hi, lo) planes staying R*cp halves apart.
    `win_dst` + `win_geom` (h, w, kh, kw, sh, sw, mask): output channels [win_c0, win_c1) go to the window-major operand
    planes of the tensor-core attention instead (see include/unimatch_sm100.h)."""
    d = ConvDesc()
    if rows:
        if rows % 16 or src0.dim() != 3 or rows > src0.shape[1]:
            raise RuntimeError("conv2d_tc: rows must be a multiple of 16 within the [2, R, cp] source planes")
        b, h, w, cp0 = 1, rows // 16, 16, src0.shape[-1]
        # the (hi, lo) planes may be row ranges of larger buffers (a slab of the token rows): distance = stride of dim 0
        d.src_plane_stride = src0.stride(0)
        if src1 is not None and (src1.shape[1] != src0.shape[1] or src1.stride(0) != src0.stride(0)):
            raise RuntimeError("conv2d_tc: both sources must have the same number of rows and the same plane stride")
        if out_split is not None:
            d.split_plane_stride = out_split.stride(0)
    else:
        _, b, h, w, cp0 = src0.shape
    d.src[0] = src0.data_ptr(); d.cin_p[0] = cp0
    d.nsrc = 1
    if src1 is not None:
        d.src[1] = src1.data_ptr(); d.cin_p[1] = src1.shape[-1]; d.nsrc = 2
    d.batch, d.h, d.w = b, h, w
    d.weights = weights.data_ptr()
    d.bias = bias.data_ptr() if bias is not None else None
    d.kh, d.kw, d.pad_h, d.pad_w = kh, kw, pad_h, pad_w
    d.stride = stride
    d.cout, d.cout_p, d.bn = cout, weights.shape[1], bn
    d.mode, d.act = mode, act
    if out_f32 is not None:
        _f32c(out_f32, "out_f32", rows_ok=True)
        d.out_f32 = out_f32.data_ptr(); d.ld_f32 = out_f32.stride(-2); d.off_f32 = off_f32
    if out_split is not None:
        d.out_split = out_split.data_ptr(); d.cp_split = out_split.shape[-1]; d.off_split = off_split
    if aux0 is not None:
        d.aux0 = aux0.data_ptr(); d.ld_aux0 = aux0.stride(-2)
    if aux1 is not None:
        d.aux1 = aux1.data_ptr(); d.ld_aux1 = aux1.stride(-2)
    if gamma is not None:
        d.gamma = gamma.data_ptr(); d.beta = beta.data_ptr()
    if pre is not None:
        _f32c(pre, "pre", rows_ok=True)
        d.pre = pre.data_ptr(); d.ld_pre = pre.stride(-2)
    if win_dst is not None:
        g = AttnGeom(*win_geom)
        lp = int(LIB.um_attention_planes_lp(ctypes.byref(g)))
        nops = (win_c1 - win_c0) // 128
        if win_dst.dtype != torch.float16 or not win_dst.is_contiguous() or lp == 0 or \
                win_dst.numel() != nops * 2 * win_streams * g.kh * g.kw * lp * 128:
            raise RuntimeError("conv2d_tc: win_dst must be contiguous fp16 planes [ops, 2, streams, windows, lp, 128]")
        d.win_dst = win_dst.data_ptr(); d.win_geom = g; d.win_lp = lp
        d.win_c0, d.win_c1, d.win_streams = win_c0, win_c1, win_streams
    _check(LIB.um_conv2d_tc(ctypes.byref(d), _stream()), "um_conv2d_tc")


conv2d_tc = _define(
    "conv2d_tc(Tensor src0, Tensor? src1, Tensor weights, Tensor? bias, int kh, int kw, int pad_h, int pad_w, int cout, "
    "int bn, int mode, int act, Tensor(a!)? out_f32, int off_f32, Tensor(b!)? out_split, int off_split, Tensor? aux0, "
    "Tensor? aux1, Tensor? gamma=None, Tensor? beta=None, int stride=1, int rows=0, Tensor(c!)? win_dst=None, "
    "int[]? win_geom=None, int win_c0=0, int win_c1=0, int win_streams=0, Tensor? pre=None) -> ()", _conv2d_tc)


def ffn_tc_supported(rows):
    """The fused FFN kernel works on pairs of 128-row tiles."""
    return rows > 0 and rows % 256 == 0


def _ffn_tc(src0, src1, w1, w2, residual, gamma, beta, out_f32, out_split, rows):
    """out = residual + LayerNorm(GELU([src0 | src1] W1^T) W2^T) over the first `rows` token rows (transformer.py:137-144).
    src0 / src1 / out_split: fp16 (hi, lo) planes [2, R, 128]; w1 / w2: prepared weight planes (prep_conv_weight);
    residual / out_f32: fp32 [R, 128]."""
    for t, name in ((src0, "src0"), (src1, "src1")):
        if t.dtype != torch.float16 or t.dim() != 3 or t.shape[0] != 2 or t.shape[-1] != 128 or t.stride(-1) != 1 or \
                t.stride(1) != 128 or rows > t.shape[1]:
            raise RuntimeError("ffn_tc: %s must be fp16 planes [2, R >= rows, 128]" % name)
    if src1.stride(0) != src0.stride(0):
        raise RuntimeError("ffn_tc: both sources must have the same plane stride")
    hidden = w1.shape[1]
    if w1.shape[0] != 2 or w1.shape[2] != 256 or tuple(w2.shape) != (2, 128, hidden) or not w1.is_contiguous() or not w2.is_contiguous():
        raise RuntimeError("ffn_tc: w1 must be [2, hidden, 256] and w2 [2, 128, hidden] prepared planes")
    d = FfnDesc()
    d.src[0] = src0.data_ptr(); d.src[1] = src1.data_ptr(); d.src_plane_stride = src0.stride(0)
    d.rows = rows; d.w1 = w1.data_ptr(); d.w2 = w2.data_ptr(); d.hidden = hidden
    if residual is not None:
        _f32c(residual, "residual", rows_ok=True)
        d.residual = residual.data_ptr(); d.ld_res = residual.stride(-2)
    d.gamma = gamma.data_ptr(); d.beta = beta.data_ptr()
    if out_f32 is not None:
        _f32c(out_f32, "out_f32", rows_ok=True)
        d.out_f32 = out_f32.data_ptr(); d.ld_f32 = out_f32.stride(-2)
    if out_split is not None:
        if out_split.dtype != torch.float16 or out_split.shape[0] != 2 or out_split.shape[-1] != 128 or out_split.stride(1) != 128:
            raise RuntimeError("ffn_tc: out_split must be fp16 planes [2, R, 128]")
        d.out_split = out_split.data_ptr(); d.split_plane_stride = out_split.stride(0)
    _check(LIB.um_ffn_tc(ctypes.byref(d), _stream()), "um_ffn_tc")


ffn_tc = _define(
    "ffn_tc(Tensor src0, Tensor src1, Tensor w1, Tensor w2, Tensor? residual, Tensor gamma, Tensor beta, "
    "Tensor(a!)? out_f32, Tensor(b!)? out_split, int rows) -> ()", _ffn_tc)


# ---- instance norm -----------------------------------------------------------------------------------------------
def _instance_norm_stats(x):
    """x: fp32 [N, h, w, C] channel-last (last dim contiguous) -> stats [N, 2, C] (mean, rstd)."""
    _f32c(x, "x", rows_ok=True)
    n, c = x.shape[0], x.shape[-1]
    hw = x[0].numel() // c
    scratch = torch.empty((int(LIB.um_instance_norm_scratch_floats(n, c)),), device=x.device, dtype=torch.float32)
    stats = torch.empty((n, 2, c), device=x.device, dtype=torch.float32)
    _check(LIB.um_instance_norm_stats(_p(x), x.stride(-2), n, hw, c, _p(scratch), _p(stats), _stream()),
           "um_instance_norm_stats")
    return stats


instance_norm_stats = _define("instance_norm_stats(Tensor x) -> Tensor", _instance_norm_stats)


def _instance_norm_apply(a, stats_a, relu_a, res, stats_res, relu_out, out_f32, out_split, off):
    _f32c(a, "a", rows_ok=True)
    n, c = a.shape[0], a.shape[-1]
    hw = a[0].numel() // c
    _check(LIB.um_instance_norm_apply(_p(a), a.stride(-2), _p(stats_a), int(relu_a), _p(res),
                                      res.stride(-2) if res is not None else 0, _p(stats_res), int(relu_out), _p(out_f32),
                                      out_f32.stride(-2) if out_f32 is not None else 0, _p(out_split),
                                      out_split.shape[-1] if out_split is not None else 0, off, n, hw, c, _stream()),
           "um_instance_norm_apply")


instance_norm_apply = _define(
    "instance_norm_apply(Tensor a, Tensor? stats_a, bool relu_a, Tensor? res, Tensor? stats_res, bool relu_out, "
    "Tensor(a!)? out_f32, Tensor(b!)? out_split, int off) -> ()", _instance_norm_apply)


# ---- 7x7 convolutions on 1-3 input channels -----------------------------------------------------------------------
def _conv7x7_small(in0, in1, nchw, weight, bias, stride, relu, scale, shift, out_f32, out_split):
    _f32c(in0, "in0"), _f32c(weight, "weight")
    if nchw:
        n0, cin, h, w = in0.shape
        n = n0 + (in1.shape[0] if in1 is not None else 0)
    else:
        n, h, w, cin = in0.shape
        n0 = n
    cout = weight.shape[0]
    sc = (ctypes.c_float * 3)(*scale) if scale is not None else None
    sh = (ctypes.c_float * 3)(*shift) if shift is not None else None
    _check(LIB.um_conv7x7_small(_p(in0), _p(in1), int(nchw), n0, n, h, w, cin, stride, _p(weight), _p(bias), cout, int(relu),
                                sc, sh, _p(out_f32), out_f32.stride(-2) if out_f32 is not None else 0, _p(out_split),
                                out_split.shape[-1] if out_split is not None else 0, _stream()), "um_conv7x7_small")


conv7x7_small = _define(
    "conv7x7_small(Tensor in0, Tensor? in1, bool nchw, Tensor weight, Tensor? bias, int stride, bool relu, float[]? scale, "
    "float[]? shift, Tensor(a!)? out_f32, Tensor(b!)? out_split) -> ()", _conv7x7_small)
