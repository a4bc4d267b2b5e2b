"""CPU reference semantics for every `torch.ops.unimatch_sm100.*` op, expressed through the ORACLE
(oracle/unimatch_oracle.py restates the reference functions; pinned by tests/golden).  Test infrastructure:

  * `-m gpu` parity tests compare each CUDA op with the function of the same name here on identical inputs;
  * `register_cpu_kernels()` installs these functions as the ops' CPU kernels *inside the test process only*,
    so the host orchestration of `unimatch_b200.UniMatch` can be checked end to end against the oracle on a
    machine without a GPU.  The product never does this: outside tests the ops have no CPU kernel.
"""
import torch

from oracle import unimatch_oracle as O
from unimatch_b200 import ops

C = 128


def _nchw(x_cl):
    return x_cl.permute(0, 3, 1, 2).contiguous()


def _cl(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous()


def window_attention(q, k, v, kv_shift, h, w, kh, kw, sh, sw, mask_mode):
    q, k, v = q.contiguous(), torch.roll(k, -kv_shift, 0).contiguous(), torch.roll(v, -kv_shift, 0).contiguous()
    shift = (sh > 0) or (sw > 0)
    assert (mask_mode == ops.MASK_SWIN) == shift
    if kh == 1 and kw == 1:
        return O.attn_full(q, k, v)
    if kh == h and kw == 1:
        return O.attn_full_1d(q, k, v, h, w)
    if kh == kw:
        wh, ww = h // kh, w // kw
        mask = O.shift_mask_2d(h, w, wh, ww, wh // 2, ww // 2, q.device) if shift else None
        if shift:
            assert sh == wh // 2 and sw == ww // 2
        return O.attn_window_2d(q, k, v, kh, shift, h, w, mask)
    assert kh == h
    ww = w // kw
    mask = O.shift_mask_1d(w, ww, ww // 2, q.device) if shift else None
    if shift:
        assert sh == 0 and sw == ww // 2
    return O.attn_window_1d(q, k, v, kw, shift, h, w, mask)


def softmax_expectation(q, k, values, n_streams, kv_shift, vdim, value_mode, post_op, h, w, kh, kw, mask_mode):
    """Dense restatement of matching.py:7-36 / :126-151 / attention.py:194-215 on token matrices."""
    n_total, L, c = q.shape
    idx = (torch.arange(n_streams) + kv_shift) % n_total
    qq, kk = q[:n_streams], k[idx]
    ys, xs = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    xs, ys = xs.reshape(-1).float(), ys.reshape(-1).float()
    if value_mode == ops.VALUE_TENSOR:
        val = values[idx]
    elif value_mode == ops.VALUE_COORDS:
        val = torch.stack([xs, ys], -1)[None].repeat(n_streams, 1, 1)
    else:
        val = xs[None, :, None].repeat(n_streams, 1, 1)
    s = torch.matmul(qq, kk.permute(0, 2, 1)) / (c ** 0.5)
    if kh == 1 and kw == 1:
        allowed = torch.ones(L, L, dtype=torch.bool)
    else:
        assert kh == h and kw == 1            # one window per image row
        allowed = (ys[:, None] == ys[None, :])
    if mask_mode == ops.MASK_CAUSAL:
        s = torch.where((xs[None, :] > xs[:, None])[None], torch.full_like(s, -1e9), s)
    s = torch.where(allowed[None], s, torch.full_like(s, float("-inf")))
    out = torch.matmul(torch.softmax(s, dim=-1), val)
    own = torch.stack([xs, ys], -1)[None]
    if post_op == ops.POST_MINUS_OWN:
        out = out - own
    elif post_op == ops.POST_OWN_MINUS:
        out = own[..., :1] - out
    return out


def local_corr_softmax(f0, f1, h, w, ry, rx, stereo):
    a, b = _nchw(f0.view(-1, h, w, C)), _nchw(f1.view(-1, h, w, C))
    if stereo:
        assert ry == 0
        return _cl(O.local_corr_disp(a, b, rx))
    assert ry == rx
    return _cl(O.local_corr_flow(a, b, rx))


def _as_flow2(flow):
    if flow.shape[-1] == 2:
        return _nchw(flow)
    d = _nchw(flow)
    return torch.cat((-d, torch.zeros_like(d)), dim=1)


def local_corr_volume(f0, f1, flow, h, w, radius):
    a, b = _nchw(f0.view(-1, h, w, C)), _nchw(f1.view(-1, h, w, C))
    return _cl(O.local_corr_volume(a, b, _as_flow2(flow), radius))


def flow_warp(f, flow, h, w):
    return _cl(O.warp_by_flow(_nchw(f.view(-1, h, w, C)), _as_flow2(flow))).view(f.shape)


def fb_consistency(fwd_flow, bwd_flow, alpha, beta):
    return O.fb_consistency(fwd_flow, bwd_flow, alpha, beta)


def propagate_local(q, k, flow, h, w, radius):
    """attention.py:217-253 with the projections already applied."""
    b = q.shape[0]
    vc = flow.shape[-1]
    ks = 2 * radius + 1
    qq = q.reshape(b * h * w, 1, C)
    kp = k.reshape(b, h, w, C).permute(0, 3, 1, 2)
    kw = torch.nn.functional.unfold(kp, kernel_size=ks, padding=radius).view(b, C, ks ** 2, h, w)
    kw = kw.permute(0, 3, 4, 1, 2).reshape(b * h * w, C, ks ** 2)
    fw = torch.nn.functional.unfold(_nchw(flow), kernel_size=ks, padding=radius).view(b, vc, ks ** 2, h, w)
    fw = fw.permute(0, 3, 4, 2, 1).reshape(b * h * w, ks ** 2, vc)
    p = torch.softmax(torch.matmul(qq, kw) / (C ** 0.5), dim=-1)
    return torch.matmul(p, fw).view(b, h, w, vc)


def depth_corr_softmax(f0, f1, K, Kinv, pose, cand, h, w, from_argmax):
    b = f0.shape[0]
    a, bb = _nchw(f0.view(b, h, w, C)), _nchw(f1.view(b, h, w, C))
    cc = cand.view(1, -1, 1, 1).repeat(b, 1, h, w)
    return _cl(O.depth_corr(a, bb, K, pose, cc, from_argmax, False))


def add_position(x, table, h, w):
    wh, ww = table.shape[0], table.shape[1]
    return x + table.repeat(h // wh, w // ww, 1)[None]


def layernorm_residual(x, residual, gamma, beta):
    y = torch.nn.functional.layer_norm(x, (C,), gamma, beta)
    return y if residual is None else residual + y


def convex_upsample(flow, mask, factor, mult):
    return O.convex_upsample(_nchw(flow), _nchw(mask), factor, is_depth=(mult == 1.0))


def upsample2x(flow, mult):
    return _cl(torch.nn.functional.interpolate(_nchw(flow), scale_factor=2, mode="bilinear", align_corners=True) * mult)


def resize_bilinear(x, h_out, w_out, scale, flip_x):
    y = torch.nn.functional.interpolate(x, size=(h_out, w_out), mode="bilinear", align_corners=True)
    if scale is not None:
        y = y * torch.tensor(list(scale)).view(1, -1, 1, 1)
    return torch.flip(y, dims=[-1]) if flip_x else y


def gru_rh(r_pre, h):
    return torch.sigmoid(r_pre) * h


def gru_update(z_pre, q_pre, h):
    z = torch.sigmoid(z_pre)
    return (1 - z) * h + z * torch.tanh(q_pre)


def split_planes(src, dst, off):
    s2 = src.reshape(-1, src.shape[-1]).float()
    hi = s2.half()
    lo = (s2 - hi.float()).half()
    rows, c = s2.shape
    d = dst.view(2, -1, dst.shape[-1])                           # dst may hold more rows than src (row padding)
    d[0, :rows, off:off + c] = hi
    d[1, :rows, off:off + c] = lo


def window_rows(h, w, kh, kw, sh, sw, lp):
    """Row (inside one stream's [windows * lp] block) of every token t = y*w + x in the window-major operand planes:
    cyclic shift (attention.py:72-79) then window split (utils.py:46-47)."""
    ys, xs = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    yr, xr = (ys - sh) % h, (xs - sw) % w
    wh, ww = h // kh, w // kw
    return (((yr // wh) * kw + xr // ww) * lp + (yr % wh) * ww + xr % ww).reshape(-1)


def planes_lp(h, w, kh, kw):
    lw = (h // kh) * (w // kw)
    return (lw + 127) // 128 * 128


def window_attention_planes(qp, kp, vp, n, kv_shift, h, w, kh, kw, sh, sw, mask_mode, out_f32, out_split):
    lp = planes_lp(h, w, kh, kw)
    rows = window_rows(h, w, kh, kw, sh, sw, lp)
    tok = lambda pl: _unsplit(pl.view(2, n, kh * kw * lp, C))[:, rows]          # [n, L, C] in token order
    out = window_attention(tok(qp), tok(kp), tok(vp), kv_shift, h, w, kh, kw, sh, sw, mask_mode)
    if out_f32 is not None:
        out_f32.copy_(out)
    if out_split is not None:
        split_planes(out.reshape(-1, C), out_split, 0)


def _unsplit(planes):
    return planes[0].float() + planes[1].float()


def instance_norm_stats(x):
    n, c = x.shape[0], x.shape[-1]
    v = x.reshape(n, -1, c).double()
    mean = v.mean(1)
    var = v.var(1, unbiased=False)
    return torch.stack([mean, 1.0 / torch.sqrt(var + 1e-5)], dim=1).float()


def instance_norm_apply(a, stats_a, relu_a, res, stats_res, relu_out, out_f32, out_split, off):
    def norm(t, st):
        if st is None:
            return t
        shp = (t.shape[0],) + (1,) * (t.dim() - 2) + (t.shape[-1],)
        return (t - st[:, 0].view(shp)) * st[:, 1].view(shp)
    y = norm(a, stats_a)
    if relu_a:
        y = torch.relu(y)
    if res is not None:
        y = y + norm(res, stats_res)
    if relu_out:
        y = torch.relu(y)
    if out_f32 is not None:
        out_f32.copy_(y)
    if out_split is not None:
        split_planes(y, out_split, off)


def conv7x7_small(in0, in1, nchw, weight, bias, stride, relu, scale, shift, out_f32, out_split):
    F = torch.nn.functional
    if nchw:
        x = in0 if in1 is None else torch.cat((in0, in1), 0)
        if scale is not None:
            x = x * torch.tensor(scale).view(1, -1, 1, 1) + torch.tensor(shift).view(1, -1, 1, 1)
    else:
        x = in0.permute(0, 3, 1, 2)
    y = F.conv2d(x, weight, bias, stride=stride, padding=3).permute(0, 2, 3, 1)
    if relu:
        y = torch.relu(y)
    if out_f32 is not None:
        out_f32.copy_(y)
    if out_split is not None:
        split_planes(y.contiguous(), out_split, 0)


def conv2d_tc(src0, src1, weights, bias, kh, kw, pad_h, pad_w, cout, bn, mode, act, out_f32, off_f32, out_split,
              off_split, aux0, aux1, gamma=None, beta=None, stride=1, rows=0, win_dst=None, win_geom=None, win_c0=0,
              win_c1=0, win_streams=0, pre=None):
    """CPU statement of um_conv2d_tc: the same fp16 (hi, lo) planes in, exact fp32 convolution of hi+lo."""
    F = torch.nn.functional
    wmat = _unsplit(weights)                                     # [cout_p, ktot]
    acc, kbase = None, 0
    for src in (src0, src1):
        if src is None:
            continue
        x = _unsplit(src)                                        # [B,h,w,cp]  (rows mode: [R, cp])
        if rows:
            x = x[:rows].reshape(1, rows // 16, 16, x.shape[-1])
        cp = x.shape[-1]
        wk = wmat[:, kbase:kbase + kh * kw * cp].view(-1, kh, kw, cp).permute(0, 3, 1, 2)
        y = F.conv2d(x.permute(0, 3, 1, 2), wk, None, stride=stride, padding=(pad_h, pad_w))
        acc = y if acc is None else acc + y
        kbase += kh * kw * cp
    full = acc.permute(0, 2, 3, 1)                               # [B,h,w,cout_p]
    y = full[..., :cout]
    if bias is not None:
        y = y + bias
    if pre is not None:
        y = y + pre[..., :cout]

    def put_f32(val, c0, c1):
        if rows:
            out_f32.view(-1, out_f32.shape[-1])[:rows, off_f32 + c0:off_f32 + c1] = val.reshape(rows, -1)
        else:
            out_f32[..., off_f32 + c0:off_f32 + c1] = val

    def put_split(val, c0):
        split_planes(val.reshape(-1, val.shape[-1]), out_split, off_split + c0)

    if mode == ops.CONV_GRU_ZR:
        y = torch.sigmoid(y)
        put_f32(y[..., :128], 0, 128)
        put_split(y[..., 128:] * aux0, 0)
        return
    if mode == ops.CONV_LN:
        y = torch.nn.functional.layer_norm(y, (128,), gamma, beta)
        if aux0 is not None:
            y = (aux0.reshape(-1, 128)[:rows].reshape(y.shape) if rows else aux0) + y
    elif mode == ops.CONV_GRU_Q:
        y = (1 - aux1) * aux0 + aux1 * torch.tanh(y)
    elif act == ops.ACT_RELU:
        y = torch.relu(y)
    elif act == ops.ACT_TANH:
        y = torch.tanh(y)
    elif act == ops.ACT_SIGMOID:
        y = torch.sigmoid(y)
    elif act == ops.ACT_GELU:
        y = torch.nn.functional.gelu(y)
    if win_dst is None:
        if out_f32 is not None:
            put_f32(y, 0, cout)
        if out_split is not None:
            put_split(y, 0)
        return
    # channels [win_c0, win_c1) -> window-major operand planes, the rest as usual
    h_, w_, kh_, kw_, sh_, sw_, _ = win_geom
    lp = planes_lp(h_, w_, kh_, kw_)
    dst_rows = window_rows(h_, w_, kh_, kw_, sh_, sw_, lp)
    L = h_ * w_
    nops = (win_c1 - win_c0) // 128
    wd = win_dst.view(nops, 2, win_streams, kh_ * kw_ * lp, 128)
    flat = full.reshape(-1, full.shape[-1])[:win_streams * L]
    if bias is not None:
        flat = flat.clone()
        flat[:, :cout] += bias
    for o in range(nops):
        v = flat[:, win_c0 + 128 * o:win_c0 + 128 * (o + 1)].reshape(win_streams, L, 128).float()
        hi = v.half()
        wd[o, 0][:, dst_rows] = hi
        wd[o, 1][:, dst_rows] = (v - hi.float()).half()
    for c0, c1 in ((0, win_c0), (win_c1, cout)):
        if c1 > c0:
            if out_f32 is not None:
                put_f32(y[..., c0:c1], c0, c1)
            if out_split is not None:
                split_planes(y[..., c0:c1].reshape(-1, c1 - c0), out_split, off_split + c0)


def ffn_tc(src0, src1, w1, w2, residual, gamma, beta, out_f32, out_split, rows):
    """CPU statement of um_ffn_tc = the two um_conv2d_tc launches it fuses (hidden planes materialised)."""
    hidden = w1.shape[1]
    hid = torch.zeros((2, src0.shape[1], hidden), dtype=torch.float16)
    conv2d_tc(src0, src1, w1, None, 1, 1, 0, 0, hidden, 256, ops.CONV_LINEAR, ops.ACT_GELU, None, 0, hid, 0, None, None,
              rows=rows)
    conv2d_tc(hid, None, w2, None, 1, 1, 0, 0, 128, 128, ops.CONV_LN, 0, out_f32, 0, out_split, 0, residual, None,
              gamma=gamma, beta=beta, rows=rows)


ALL = ["split_planes", "conv7x7_small", "conv2d_tc", "ffn_tc", "instance_norm_stats", "instance_norm_apply", "window_attention", "window_attention_planes", "softmax_expectation", "local_corr_softmax", "local_corr_volume", "flow_warp", "fb_consistency",
       "propagate_local", "depth_corr_softmax", "add_position", "layernorm_residual", "convex_upsample", "upsample2x", "resize_bilinear",
       "gru_rh", "gru_update"]

_registered = []


def register_cpu_kernels():
    """Install the functions above as CPU kernels of the unimatch_sm100 ops (tests only)."""
    if _registered:
        return
    lib = torch.library.Library("unimatch_sm100", "IMPL", "CPU")
    g = globals()
    for name in ALL:
        lib.impl(name, g[name])
    _registered.append(lib)


def unregister_cpu_kernels():
    """Remove the CPU kernels installed by `register_cpu_kernels()`: the ops are back to the product's, which have none."""
    while _registered:
        _registered.pop()._destroy()
