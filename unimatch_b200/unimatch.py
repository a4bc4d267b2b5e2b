"""Drop-in `UniMatch(nn.Module)`: the reference's constructor, `forward()` signature, `state_dict` layout and
`{'flow_preds': [...]}` output (reference `unimatch/unimatch.py:17-26, :95-111, :365-367`), with the matching
path executed by libunimatch_sm100 (hand-written sm_100a kernels) instead of eager PyTorch ops.

Host side = plain PyTorch orchestration:
  * parameters live in a module tree generated from `spec.param_spec` (same keys/shapes as the reference);
  * activations are channel-last end to end: feature maps are token matrices [N, L=h*w, 128] (N = 2 x pairs:
    all first views, then all second views), flow-like maps are [B, h, w, F];
  * `concat1` of the reference transformer (transformer.py:271-286) is never materialised: the cross-attention
    kernel reads keys/values of the partner stream (n + N/2) mod N;
  * loop-invariant / dead work of the refinement loop is hoisted (`refine_proj`, unimatch.py:315-320) or skipped
    (mask head on non-final iterations, unimatch.py:333,351) -- results are unchanged.
Every Linear layer, the CNN backbone, the update-block convolutions, the `upsampler` head and the propagation
projections run on the library's tcgen05 implicit-GEMM kernel (`um_conv2d_tc`, fp32-faithful split-fp16 operands);
attention / correlation on the tcgen05 attention kernels.  There is no cuDNN / cuBLAS call on the path and no
alternative backend in this module (A/B harnesses against the libraries live in tools/ab_paths.py).

The forward pass is a sequence of `_stage_*` methods (encoder, position + warp, transformer, correlation,
propagation, refinement iteration, upsampling) so that the parity tests can teacher-force every stage with the
oracle's intermediate tensors at the BASELINE shapes (tests/test_stages_gpu.py).

Inference only (the reference's callers use eval()/no_grad, evaluate_flow.py:19,33); `train()` mode raises.
"""
import math
from contextlib import contextmanager

import torch
import torch.nn as nn

from . import ops
from .spec import param_spec

_OPS = torch.ops.unimatch_sm100


import os as _os
_FUSED_FFN = _os.environ.get("UM_FUSED_FFN", "1") != "0"      # A/B switch of the fused FFN kernel (tools / profiling)
_CORR_TC = _os.environ.get("UM_CORR_TC", "1") != "0"          # A/B switch of the tensor-core correlation volume (tools / profiling)


def _bn256(b, h, w):
    """Output-channel tile of the 256-channel update-block convolutions (GRU z|r, flow / mask heads).  With an even number of
    16 x 8 pixel tiles the launch runs on CTA pairs (um_conv_tc.cu, PAIR): two 128-wide tiles with double-buffered TMEM
    accumulators (the epilogue overlaps the next tile's MMAs; measured 16.3 -> 15.3 ms per step for the update block) beat
    one 256-wide tile with a single buffer.  A lone CTA reads its A tile once per channel tile: the wide tile wins there."""
    return 128 if (b * ((h + 7) // 8) * ((w + 15) // 16)) % 2 == 0 else 256



class _Node(nn.Module):
    """Parameter container; gives the flat spec table the reference's dotted state_dict names."""


def _attach(root, key, param):
    parts = key.split(".")
    node = root
    for name in parts[:-1]:
        if name not in node._modules:
            node.add_module(name, _Node())
        node = node._modules[name]
    node.register_parameter(parts[-1], param)


def _sine_table(wh, ww):
    """PositionEmbeddingSine on a wh x ww window (position.py:26-45) as a [wh, ww, 128] table:
    channels 0..63 encode y, 64..127 encode x; sin on even, cos on odd feature indices."""
    y = torch.arange(1, wh + 1, dtype=torch.float32)
    x = torch.arange(1, ww + 1, dtype=torch.float32)
    y = y / (float(wh) + 1e-6) * (2 * math.pi)
    x = x / (float(ww) + 1e-6) * (2 * math.pi)
    n = torch.arange(64, dtype=torch.float32)
    dim_t = 10000 ** (2 * torch.div(n, 2, rounding_mode="floor") / 64)
    even = (torch.arange(64) % 2 == 0)

    def enc(v):
        a = v[:, None] / dim_t
        return torch.where(even, a.sin(), a.cos())

    ey, ex = enc(y), enc(x)
    return torch.cat((ey[:, None, :].expand(wh, ww, 64), ex[None, :, :].expand(wh, ww, 64)), dim=2).contiguous()


def _ceil16(n):
    return (n + 15) // 16 * 16


class UniMatch(nn.Module):
    def __init__(self, num_scales=1, feature_channels=128, upsample_factor=8, num_head=1, ffn_dim_expansion=4,
                 num_transformer_layers=6, reg_refine=False, task="flow"):
        super().__init__()
        if feature_channels != 128:
            raise ValueError("libunimatch_sm100 is built for feature_channels=128 (main_flow.py:73)")
        if num_head != 1:
            raise NotImplementedError("multi-head attention is not implemented (as in transformer.py:63-66)")
        self.feature_channels = feature_channels
        self.num_scales = num_scales
        self.upsample_factor = upsample_factor
        self.reg_refine = reg_refine
        self.num_transformer_layers = num_transformer_layers
        self.task_built = task
        self._spec = param_spec(num_scales, feature_channels, upsample_factor, num_head, ffn_dim_expansion,
                                num_transformer_layers, reg_refine, task)
        for key, shape in self._spec.items():
            _attach(self, key, nn.Parameter(self._init_tensor(key, shape)))
        self._prep_key = None
        self._prep = None
        self._tables = {}
        self._attn_ws = {}           # window-major attention operand planes, cached per (device, streams, geometry)
        self._pad_ws = {}            # zero-padded plane buffers, cached per (use, shape)
        self.training = False        # inference-only module: starts (and stays) in eval mode
        self.kernel_timer = None     # bench hook: dict -> CUDA-event pairs around launch groups

    @staticmethod
    def _init_tensor(key, shape):
        # same families as the reference initialisers (backbone.py:88-95, transformer.py:222-224, attention.py:180-182)
        t = torch.empty(shape)
        if len(shape) == 4:
            nn.init.kaiming_normal_(t, mode="fan_out", nonlinearity="relu")
        elif len(shape) == 2:
            nn.init.xavier_uniform_(t)
        elif ".norm" in key:
            t.fill_(1.0 if key.endswith("weight") else 0.0)
        else:
            t.uniform_(-0.05, 0.05)
        return t

    def train(self, mode=True):
        if mode:
            raise NotImplementedError("unimatch_b200.UniMatch is inference-only (use .eval(); training stays on the reference)")
        return super().train(False)

    # ------------------------------------------------------------------------------------------ weights
    def _prepared(self):
        """fp16 (hi, lo) weight planes of every layer (`ops.prep_conv_weight`), rebuilt when a parameter changes."""
        params = dict(self.named_parameters())
        key = (tuple((p._version, p.data_ptr()) for p in params.values()),)
        if self._prep_key == key:
            return self._prep
        w = {k: v.detach() for k, v in params.items()}
        prep = ops.prep_conv_weight
        lin = lambda m: m[:, :, None, None]
        P = {"raw": w, "blocks": []}
        for i in range(self.num_transformer_layers):
            sk, ck = "transformer.layers.%d.self_attn." % i, "transformer.layers.%d.cross_attn_ffn." % i
            w_in = torch.cat([w[sk + "q_proj.weight"], w[sk + "k_proj.weight"], w[sk + "v_proj.weight"],
                              w[ck + "k_proj.weight"], w[ck + "v_proj.weight"]], dim=0)        # [640, 128]
            hid = w[ck + "mlp.0.weight"].shape[0]
            P["blocks"].append(dict(
                tc_in=prep(lin(w_in), [128], 640),
                tc_m_s=prep(lin(w[sk + "merge.weight"]), [128], 128), g_s=w[sk + "norm1.weight"], b_s=w[sk + "norm1.bias"],
                tc_q_c=prep(lin(w[ck + "q_proj.weight"]), [128], 128),
                tc_m_c=prep(lin(w[ck + "merge.weight"]), [128], 128), g_c1=w[ck + "norm1.weight"], b_c1=w[ck + "norm1.bias"],
                tc_w1=prep(lin(w[ck + "mlp.0.weight"]), [128, 128], hid),
                tc_w2=prep(lin(w[ck + "mlp.2.weight"]), [hid], 128), g_c2=w[ck + "norm2.weight"], b_c2=w[ck + "norm2.bias"],
                hid=hid))
        P["tcb"] = self._prepare_backbone(w)
        # SelfAttnPropagation projections (attention.py:177-178, :204-205, :227-232)
        qw, qb = w["feature_flow_attn.q_proj.weight"], w["feature_flow_attn.q_proj.bias"]
        kw, kb = w["feature_flow_attn.k_proj.weight"], w["feature_flow_attn.k_proj.bias"]
        P["prop_q"] = (prep(lin(qw), [128], 128), qb.contiguous())
        P["prop_k"] = (prep(lin(kw), [128], 128), kb.contiguous())
        P["prop_qk"] = (prep(lin(torch.cat([qw, kw], 0)), [128], 256), torch.cat([qb, kb]).contiguous())
        if self.reg_refine:
            P["tc"] = self._prepare_refine(w)
        if "upsampler.0.weight" in w:                                           # unimatch.py:47-52
            w0 = w["upsampler.0.weight"]                                        # [256, 2 + 128, 3, 3], input = cat(flow, feature)
            w0 = torch.cat([w0[:, 2:], w0[:, :2]], dim=1)                       # our planes hold [feature | flow]
            nm = w["upsampler.2.weight"].shape[0]
            bn2 = 192 if nm % 192 == 0 else 64
            P["up"] = dict(c0=(prep(w0, [130], 256), w["upsampler.0.bias"]),
                           c2=(prep(w["upsampler.2.weight"], [256], (nm + bn2 - 1) // bn2 * bn2), w["upsampler.2.bias"]),
                           nm=nm, bn2=bn2)
        self._prep_key, self._prep = key, P
        return P

    @staticmethod
    def _prepare_backbone(w):
        """fp16 (hi, lo) weight planes of the CNN encoder convolutions (backbone.py:49-86) for um_conv2d_tc."""
        T = {}
        for key, wt in w.items():
            if not key.startswith("backbone.") or not key.endswith(".weight") or key == "backbone.conv1.weight":
                continue
            cout, cin = wt.shape[0], wt.shape[1]
            bn = 128 if cout > 64 else 64          # 96 channels: one padded 128-wide tile beats two 64-wide (A is read once)
            T[key[:-7]] = (ops.prep_conv_weight(wt, [cin], (cout + bn - 1) // bn * bn), w.get(key[:-7] + ".bias"), bn)
        return T

    @staticmethod
    def _prepare_refine(w):
        """fp16 (hi, lo) weight planes for um_conv2d_tc, K ordered (source, tap, ci); see ops.prep_conv_weight."""
        prep = ops.prep_conv_weight
        fd = w["refine.flow_head.conv2.weight"].shape[0]
        T = {"fd": fd}
        pw, pb = w["refine_proj.weight"], w["refine_proj.bias"]
        T["proj_net"] = (prep(pw[:128], [128], 128), pb[:128].contiguous())
        T["proj_inp"] = (prep(pw[128:], [128], 128), pb[128:].contiguous())
        e = "refine.encoder."
        T["convc1"] = (prep(w[e + "convc1.weight"], [81], 256), w[e + "convc1.bias"])
        T["convc2"] = (prep(w[e + "convc2.weight"], [256], 192), w[e + "convc2.bias"])
        T["convf2"] = (prep(w[e + "convf2.weight"], [128], 64), w[e + "convf2.bias"])
        T["conv"] = (prep(w[e + "conv.weight"], [256], 128), w[e + "conv.bias"])
        # SepConvGRU (reg_refine.py:22-52) over hx = cat[h, inp, motion | flow] (128 + 128 + 128 channels).  `inp` is the same in
        # every refinement iteration and so is `h` of the first half (net is not carried between iterations, unimatch.py:315-333):
        # their share of each convolution is computed ONCE per forward ("_fix" weights -> a fp32 tensor the per-iteration
        # convolution adds to its accumulator) and only the channels that changed are convolved per iteration ("_var").
        g = "refine.gru.conv"
        for sfx in ("1", "2"):
            wzr = torch.cat([w[g + "z%s.weight" % sfx], w[g + "r%s.weight" % sfx]], 0)           # [256, 384, kh, kw]
            bzr = torch.cat([w[g + "z%s.bias" % sfx], w[g + "r%s.bias" % sfx]])
            wq, bq = w[g + "q%s.weight" % sfx], w[g + "q%s.bias" % sfx]                           # [128, 384, kh, kw]
            if sfx == "1":
                T["zr1_fix"] = (prep(wzr[:, :256], [128, 128], 256), bzr)                         # h0 | inp
                T["zr1_var"] = prep(wzr[:, 256:], [128], 256)                                     # motion | flow
            else:
                T["zr2_fix"] = (prep(wzr[:, 128:256], [128], 256), bzr)                           # inp
                T["zr2_var"] = prep(torch.cat([wzr[:, :128], wzr[:, 256:]], 1), [128, 128], 256)  # h1 | motion
            T["q%s_fix" % sfx] = (prep(wq[:, 128:256], [128], 128), bq)                           # inp
            T["q%s_var" % sfx] = prep(torch.cat([wq[:, :128], wq[:, 256:]], 1), [128, 128], 128)  # r*h | motion
        T["fh1"] = (prep(w["refine.flow_head.conv1.weight"], [128], 256), w["refine.flow_head.conv1.bias"])
        T["fh2"] = (prep(w["refine.flow_head.conv2.weight"], [256], 16), w["refine.flow_head.conv2.bias"])
        if "refine.mask.0.weight" in w:
            T["mask0"] = (prep(w["refine.mask.0.weight"], [128], 256), w["refine.mask.0.bias"])
            nm = w["refine.mask.2.weight"].shape[0]
            T["mask2"] = (prep(w["refine.mask.2.weight"], [256], (nm + 63) // 64 * 64), w["refine.mask.2.bias"])
        return T

    def _pos_table(self, wh, ww, device):
        k = (wh, ww, str(device))
        if k not in self._tables:
            self._tables[k] = _sine_table(wh, ww).to(device)
        return self._tables[k]

    # ------------------------------------------------------------------------------------------ timers (bench hooks)
    @contextmanager
    def _section(self, name):
        t = self.kernel_timer
        if t is None:
            yield
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        yield
        e1.record()
        t.setdefault("_events", []).append(("sec:" + name, e0, e1, 0.0))

    def _timed(self, tag, flops, fn, *a):
        """bench hook: CUDA events around one launch group + its algorithmic FLOPs (no effect without a timer)."""
        t = self.kernel_timer
        if t is None:
            return fn(*a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn(*a)
        e1.record()
        t.setdefault("_events", []).append((tag, e0, e1, flops))
        return out

    def _conv(self, src0, src1, weights, bias, kh, kw, ph, pw, cout, *rest, **kwargs):
        """um_conv2d_tc; under the bench timer also records 2 x output pixels x cout x real K as the layer's algorithmic FLOPs."""
        if self.kernel_timer is None:
            return _OPS.conv2d_tc(src0, src1, weights, bias, kh, kw, ph, pw, cout, *rest, **kwargs)
        stride = rest[11] if len(rest) > 11 else 1
        rows = rest[12] if len(rest) > 12 else 0
        if rows:
            pix = rows
        else:
            _, b, h, w, _ = src0.shape
            pix = b * ((h + 2 * ph - kh) // stride + 1) * ((w + 2 * pw - kw) // stride + 1)
        flops = 2.0 * pix * cout * getattr(weights, "k_true", kh * kw * src0.shape[-1])
        return self._timed("conv", flops, lambda: _OPS.conv2d_tc(src0, src1, weights, bias, kh, kw, ph, pw, cout, *rest, **kwargs))

    # ------------------------------------------------------------------------------------------ backbone
    def _stage_backbone(self, P, img0, img1, normalise):
        """CNNEncoder (backbone.py:104-133) with every 3x3 / 1x1 convolution on the tcgen05 implicit-GEMM kernel and
        InstanceNorm + ReLU + residual as fused bandwidth passes that emit the next convolution's fp16 planes.
        The 7x7 stem (3 input channels) is the direct fp32 kernel `um_conv7x7_small` with `normalize_img` folded into its load.
        Returns the feature maps low -> high resolution, each [2B, h, w, 128] (first views, then second views)."""
        T = P["tcb"]
        dev = img0.device
        nb = img0.shape[0] + img1.shape[0]
        C, IS, IA = self._conv, _OPS.instance_norm_stats, _OPS.instance_norm_apply
        pad64 = lambda c: (c + 63) // 64 * 64

        nplanes = [0]

        def planes(h, w, c):
            cp = pad64(c)
            if cp == c:
                return torch.empty((2, nb, h, w, cp), device=dev, dtype=torch.float16)
            nplanes[0] += 1                                  # distinct live buffers of one forward get distinct cache slots
            return self._zero_padded("backbone%d" % nplanes[0], (2, nb, h, w, cp), dev)

        def conv(src_s, name, k, stride, cout, hw_in):
            wt, bias, bn = T[name]
            h, w = hw_in
            ho, wo = (h + 2 * (k // 2) - k) // stride + 1, (w + 2 * (k // 2) - k) // stride + 1
            out = torch.empty((nb, ho, wo, cout), device=dev)
            C(src_s, None, wt, bias, k, k, k // 2, k // 2, cout, bn, ops.CONV_LINEAR, ops.ACT_NONE, out, 0, None, 0, None,
              None, None, None, stride)
            return out

        hh, ww = img0.shape[2], img0.shape[3]
        a = torch.empty((nb, (hh - 1) // 2 + 1, (ww - 1) // 2 + 1, 64), device=dev)
        if normalise:                                        # normalize_img (utils.py:23-31) folded into the stem's load
            mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
            scale = [1.0 / (255.0 * s_) for s_ in std]
            shift = [-m_ / s_ for m_, s_ in zip(mean, std)]
        else:
            scale = shift = None
        _OPS.conv7x7_small(img0, img1, True, P["raw"]["backbone.conv1.weight"], None, 2, False, scale, shift, a, None)
        h, w = a.shape[1], a.shape[2]
        cur_f = torch.empty((nb, h, w, 64), device=dev)
        cur_s = planes(h, w, 64)
        IA(a, IS(a), True, None, None, False, cur_f, cur_s, 0)
        for li, cout, stride in ((1, 64, 1), (2, 96, 2), (3, 128, 2 if self.num_scales == 1 else 1)):
            for bi in range(2):
                pf = "backbone.layer%d.%d." % (li, bi)
                st = stride if bi == 0 else 1
                a1 = conv(cur_s, pf + "conv1", 3, st, cout, (h, w))
                ho, wo = a1.shape[1], a1.shape[2]
                t_s = planes(ho, wo, cout)
                IA(a1, IS(a1), True, None, None, False, None, t_s, 0)
                a2 = conv(t_s, pf + "conv2", 3, 1, cout, (ho, wo))
                if (pf + "downsample.0") in T:
                    res = conv(cur_s, pf + "downsample.0", 1, st, cout, (h, w))
                    st_res = IS(res)
                else:
                    res, st_res = cur_f, None
                out_f = torch.empty((nb, ho, wo, cout), device=dev)
                out_s = planes(ho, wo, cout)
                IA(a2, IS(a2), True, res, st_res, True, out_f, out_s, 0)
                cur_f, cur_s, h, w = out_f, out_s, ho, wo
        wt, bias, bn = T["backbone.conv2"]
        x6 = torch.empty((nb, h, w, 128), device=dev)
        x6_s = planes(h, w, 128) if self.num_scales > 1 else None
        C(cur_s, None, wt, bias, 1, 1, 0, 0, 128, bn, ops.CONV_LINEAR, ops.ACT_NONE, x6, 0, x6_s, 0, None, None)
        if self.num_scales == 1:
            return [x6]
        strides = (1, 2, 4, 8)[:self.num_scales]                               # trident_conv.py:64-70
        feats = [conv(x6_s, "backbone.trident_conv", 3, s, 128, (h, w)) for s in strides]
        return feats[::-1]

    # ------------------------------------------------------------------------------------------ transformer
    @staticmethod
    def _attn_plan(attn_type, splits, h, w, layer_idx):
        """(self geometry, cross geometry) as (kh, kw, sh, sw, mask) -- the dispatch of transformer.py:62-135,
        decided statically per call site instead of the reference's data-dependent `is_self_attn` sync (:55)."""
        shift = ("swin" in attn_type) and splits > 1 and layer_idx % 2 == 1
        full2d = (1, 1, 0, 0, ops.MASK_NONE)
        if splits > 1:
            wh, ww = h // splits, w // splits
            swin2d = (splits, splits, wh // 2 if shift else 0, ww // 2 if shift else 0,
                      ops.MASK_SWIN if shift else ops.MASK_NONE)
            swin1d = (h, splits, 0, ww // 2 if shift else 0, ops.MASK_SWIN if shift else ops.MASK_NONE)
        full1d = (h, 1, 0, 0, ops.MASK_NONE)
        if attn_type == "swin" and splits > 1:
            return swin2d, swin2d
        if attn_type == "self_swin2d_cross_1d":
            return (swin2d if splits > 1 else full2d), full1d
        if attn_type == "self_swin2d_cross_swin1d":
            return (swin2d if splits > 1 else full2d), (swin1d if splits > 1 else full1d)
        return full2d, full2d

    def _zero_padded(self, tag, shape, dev):
        """fp16 plane buffer whose padding channels must read as zero (e.g. 96 -> 128, 81 -> 128 channels): zero-filled once
        and cached per (use, shape) -- the kernels only ever write the real channels, so the padding stays zero and the
        per-forward fills (6 x 200 MB at the bench shape) disappear."""
        key = (tag, tuple(shape), str(dev))
        buf = self._pad_ws.get(key)
        if buf is None:
            if len(self._pad_ws) >= 24:
                self._pad_ws.clear()
            buf = torch.zeros(shape, device=dev, dtype=torch.float16)
            self._pad_ws[key] = buf
        return buf

    def _attn_planes(self, dev, n, h, w, kh, kw, lp):
        """Window-major operand planes [6 operands: q k v (self) | k v (cross) | q (cross)][2][n][windows][lp][128], zeroed once:
        the producers only ever write rows < lw of a window, so the padding rows stay zero across layers and calls."""
        key = (str(dev), n, h, w, kh, kw, lp)
        buf = self._attn_ws.get(key)
        if buf is None:
            if len(self._attn_ws) >= 4:                   # a handful of (scale, batch) shapes; do not hoard HBM beyond that
                self._attn_ws.clear()
            buf = torch.zeros((6, 2, n, kh * kw, lp, 128), device=dev, dtype=torch.float16)
            self._attn_ws[key] = buf
        return buf

    def _stage_transformer(self, P, x, h, w, attn_type, splits, tag="s0"):
        """FeatureTransformer.forward (transformer.py:226-294) on tokens x [N, L, 128], N = 2 x pairs.  Every Linear is a
        tcgen05 GEMM over token rows (activations travel as fp16 (hi, lo) planes [2, rows, C] between GEMMs); LayerNorm
        (+residual) / GELU are GEMM epilogues; `cat([source, message])` of the FFN (transformer.py:141) is a second GEMM
        source.  Where the window geometry runs on the tensor-core attention kernel, the q|k|v projections write the
        kernel's window-major operand planes directly (no fp32 q/k/v, no split pass) and the attention writes the merge
        layer's operand planes.  Returns (tokens fp32 [N, L, 128], their fp16 planes [2, rows_padded, 128])."""
        n, l, c = x.shape
        half = n // 2
        rows = n * l
        rp = _ceil16(rows)
        dev = x.device
        G, LN, LIN, NONE = self._conv, ops.CONV_LN, ops.CONV_LINEAR, ops.ACT_NONE
        mk = torch.empty if rp == rows else torch.zeros
        planes = lambda cp: mk((2, rp, cp), device=dev, dtype=torch.float16)
        f32 = lambda cols: mk((rp, cols), device=dev)
        tok = lambda t, c0, c1: t[:rows].view(n, l, t.shape[-1])[:, :, c0:c1]
        hid = P["blocks"][0]["hid"]
        x_f, xo_f, x1_f = f32(c), f32(c), f32(c)
        x_s, xo_s, x1_s, msg_s, m_s = planes(c), planes(c), planes(c), planes(c), planes(c)
        # FFN: one fused CTA-pair kernel (the 1024-wide hidden activation stays in tensor memory) when the rows are a whole
        # number of tile pairs; else two GEMM launches around hidden planes in HBM
        fused_ffn = _FUSED_FFN and ops.ffn_tc_supported(rp)
        hid_s = None if fused_ffn else planes(hid)
        x_f[:rows] = x.reshape(rows, c)
        _OPS.split_planes(x_f, x_s, 0)
        y = q_f = None
        for i, blk in enumerate(P["blocks"]):
            geo_s, geo_c = self._attn_plan(attn_type, splits, h, w, i)
            gs, gc = (h, w) + geo_s, (h, w) + geo_c
            lp_s = ops.attention_planes_lp(*gs)
            lp_c = ops.attention_planes_lp(*gc) if geo_c == geo_s else 0      # cross planes only when they share the buffers
            ws = self._attn_planes(dev, n, h, w, geo_s[0], geo_s[1], lp_s) if lp_s else None
            # ---- q_s | k_s | v_s | k_c | v_c = x W_in^T
            win_c1 = 640 if lp_c else (384 if lp_s else 0)
            if win_c1 < 640 and y is None:
                y = f32(5 * c)
            G(x_s, None, blk["tc_in"], None, 1, 1, 0, 0, 5 * c, 128, LIN, NONE, y if win_c1 < 640 else None, 0, None, 0, None,
              None, None, None, 1, rp, ws[:win_c1 // 128] if win_c1 else None, gs if win_c1 else None, 0, win_c1, n)
            # ---- self-attention -> merge + LayerNorm + residual (transformer.py:137-144, no FFN: :157-161)
            fl_s, fl_c = (4.0 * (l // (g[0] * g[1])) * l * 128 * n for g in (geo_s, geo_c))   # 4 Lw^2 C per window per stream
            if lp_s:
                self._timed("attn:" + tag, fl_s, _OPS.window_attention_planes, ws[0], ws[1], ws[2], n, 0, *gs, None, msg_s)
            else:
                msg = self._timed("attn_simt:" + tag, fl_s, _OPS.window_attention, tok(y, 0, 128), tok(y, 128, 256), tok(y, 256, 384), 0, *gs)
                _OPS.split_planes(msg.view(rows, c), msg_s, 0)
            G(msg_s, None, blk["tc_m_s"], None, 1, 1, 0, 0, c, 128, LN, 0, x1_f, 0, x1_s, 0, x_f, None, blk["g_s"], blk["b_s"], 1, rp)
            # ---- cross-attention: q from the updated stream, k / v from the partner stream's projections
            if lp_c:
                G(x1_s, None, blk["tc_q_c"], None, 1, 1, 0, 0, c, 128, LIN, NONE, None, 0, None, 0, None, None, None, None, 1, rp,
                  ws[5:6], gc, 0, 128, n)
                self._timed("attn:" + tag, fl_c, _OPS.window_attention_planes, ws[5], ws[3], ws[4], n, half, *gc, None, msg_s)
            else:
                if q_f is None:
                    q_f = f32(c)
                G(x1_s, None, blk["tc_q_c"], None, 1, 1, 0, 0, c, 128, LIN, NONE, q_f, 0, None, 0, None, None, None, None, 1, rp)
                msg = self._timed("attn_simt:" + tag, fl_c, _OPS.window_attention, tok(q_f, 0, 128), tok(y, 384, 512), tok(y, 512, 640), half, *gc)
                _OPS.split_planes(msg.view(rows, c), msg_s, 0)
            G(msg_s, None, blk["tc_m_c"], None, 1, 1, 0, 0, c, 128, LN, 0, None, 0, m_s, 0, None, None, blk["g_c1"], blk["b_c1"], 1, rp)
            # ---- FFN on cat([source, message]) + LayerNorm + residual
            # (Measured and not kept: FFN1 / FFN2 slab by slab over a hidden buffer that fits the L2 -- 22 x 2 launches of 71
            # CTA-pair tiles instead of 2: transformer_s1 15.0 -> 18.5 ms; launch gaps and partial waves cost more than the
            # 3.2 GB round trip of the hidden planes.)
            if fused_ffn:
                self._timed("conv", 2.0 * rp * hid * (2 * c + c), _OPS.ffn_tc, x1_s, m_s, blk["tc_w1"], blk["tc_w2"], x1_f,
                            blk["g_c2"], blk["b_c2"], xo_f, xo_s, rp)
            else:
                G(x1_s, m_s, blk["tc_w1"], None, 1, 1, 0, 0, hid, 256, LIN, ops.ACT_GELU, None, 0, hid_s, 0, None, None, None, None, 1, rp)
                G(hid_s, None, blk["tc_w2"], None, 1, 1, 0, 0, c, 128, LN, 0, xo_f, 0, xo_s, 0, x1_f, None, blk["g_c2"], blk["b_c2"], 1, rp)
            x_f, xo_f, x_s, xo_s = xo_f, x_f, xo_s, x_s
        return x_f[:rows].view(n, l, c), x_s

    # ------------------------------------------------------------------------------------------ per-scale stages
    def _stage_features(self, f0, f1, flow, h, wd, splits):
        """Warp the second view with the current estimate (unimatch.py:156-168, geometry.py:65-72) and add the per-window
        sine position encoding to both views (utils.py:111-131).  f0, f1: [Bp, h, w, 128]; returns tokens [2Bp, L, 128]."""
        Bp, c = f0.shape[0], f0.shape[-1]
        if flow is not None:
            f1 = _OPS.flow_warp(f1.contiguous(), flow.contiguous(), h, wd)
        table = self._pos_table(h // splits, wd // splits, f0.device)
        tok = torch.cat((f0, f1), dim=0).view(2 * Bp, h, wd, c)
        return _OPS.add_position(tok, table, h, wd).view(2 * Bp, h * wd, c)

    def _stage_correlation(self, tok, Bp, h, wd, task, radius, pred_bidir_flow=False, depth=None):
        """Correlation + softmax (unimatch.py:186-216) on the transformer outputs tok [2Bp, L, 128] -> [ns, h, w, fd]."""
        dev = tok.device
        t0, t1 = tok[:Bp], tok[Bp:]
        if task == "depth":
            Ks, pose, min_depth, max_depth, ncand, from_argmax, bidir = depth
            cand = torch.linspace(min_depth, max_depth, ncand).float().to(dev)                         # :190
            if bidir:
                q0, q1 = torch.cat((t0, t1), 0).contiguous(), torch.cat((t1, t0), 0).contiguous()
                Kc = Ks.repeat(2, 1, 1)
                pc = torch.cat((pose, torch.inverse(pose)), dim=0).float()
            else:
                q0, q1, Kc, pc = t0.contiguous(), t1.contiguous(), Ks, pose.float()
            return _OPS.depth_corr_softmax(q0, q1, Kc.contiguous(), torch.inverse(Kc).contiguous(), pc.contiguous(), cand,
                                           h, wd, bool(from_argmax))
        if radius == -1:
            if task == "flow":
                ns = 2 * Bp if pred_bidir_flow else Bp
                return _OPS.softmax_expectation(tok, tok, None, ns, Bp, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN,
                                                h, wd, 1, 1, ops.MASK_NONE).view(ns, h, wd, 2)
            if task == "stereo":
                return _OPS.softmax_expectation(tok, tok, None, Bp, Bp, 1, ops.VALUE_XCOORD, ops.POST_OWN_MINUS,
                                                h, wd, h, 1, ops.MASK_CAUSAL).view(Bp, h, wd, 1)
            raise NotImplementedError
        if task == "flow":
            return _OPS.local_corr_softmax(t0.contiguous(), t1.contiguous(), h, wd, radius, radius, False)
        if task == "stereo":
            return _OPS.local_corr_softmax(t0.contiguous(), t1.contiguous(), h, wd, 0, radius, True)
        raise NotImplementedError

    def _stage_propagation(self, P, x_s, flow, nb, h, wd, prop_r):
        """SelfAttnPropagation.forward (attention.py:184-253) on the first `nb` streams of the transformer output planes
        x_s [2, rows_padded, 128]: q = Wq x + bq; global: k = Wk q + bk, out = softmax(q k^T / sqrt(C)) flow;
        local (radius r): k = Wk x + bk, 3x3 zero-padded window.  Both projections are tcgen05 GEMMs."""
        dev = flow.device
        L = h * wd
        rows = nb * L
        rq = rows if rows % 16 == 0 else x_s.shape[1]            # the GEMM runs over a multiple of 16 rows
        G, LIN, NONE = self._conv, ops.CONV_LINEAR, ops.ACT_NONE
        fd = flow.shape[-1]
        flow = flow.contiguous()
        if prop_r > 0:
            qk = torch.empty((rq, 256), device=dev)
            G(x_s, None, *P["prop_qk"], 1, 1, 0, 0, 256, 128, LIN, NONE, qk, 0, None, 0, None, None, None, None, 1, rq)
            qk = qk[:rows].view(nb, L, 256)
            return _OPS.propagate_local(qk[:, :, :128], qk[:, :, 128:], flow, h, wd, prop_r)
        q = torch.empty((rq, 128), device=dev)
        q_s = torch.empty((2, rq, 128), device=dev, dtype=torch.float16)
        k = torch.empty((rq, 128), device=dev)
        G(x_s, None, *P["prop_q"], 1, 1, 0, 0, 128, 128, LIN, NONE, q, 0, q_s, 0, None, None, None, None, 1, rq)
        G(q_s, None, *P["prop_k"], 1, 1, 0, 0, 128, 128, LIN, NONE, k, 0, None, 0, None, None, None, None, 1, rq)
        return _OPS.softmax_expectation(q[:rows].view(nb, L, 128), k[:rows].view(nb, L, 128), flow.view(nb, L, fd), nb, 0, fd,
                                        ops.VALUE_TENSOR, ops.POST_NONE, h, wd, 1, 1, ops.MASK_NONE).view(nb, h, wd, fd)

    # ------------------------------------------------------------------------------------------ refinement
    class _RefineState:
        pass

    def _stage_refine_setup(self, P, feat0, b, h, w):
        """Loop-invariant part of the refinement (unimatch.py:315-320): net = tanh(.), inp = relu(.) of refine_proj(feature0),
        and the activation planes the update block reuses every iteration.  feat0: [b, h, w, 128] fp32."""
        T = P["tc"]
        dev = feat0.device
        st = self._RefineState()
        z16 = lambda cp: torch.empty((2, b, h, w, cp), device=dev, dtype=torch.float16)
        st.corr_s = self._zero_padded("corr", (2, b, h, w, 128), dev)    # 81 real channels, padding stays zero
        st.cor1_s, st.cf_s, st.flo1_s = z16(256), z16(256), z16(128)
        st.inp_s, st.mfx_s = z16(128), z16(128)                      # inp | (motion features, flow): x of the GRU in two buffers
        st.h0_s, st.h1_s, st.h2_s, st.rh_s, st.fh_s = z16(128), z16(128), z16(128), z16(128), z16(256)
        f0_s = z16(128)
        _OPS.split_planes(feat0, f0_s, 0)
        f32 = lambda cc: torch.empty((b, h, w, cc), device=dev)
        st.net0, st.z, st.h1, st.h2 = f32(128), f32(128), f32(128), f32(128)
        C, LIN, NONE = self._conv, ops.CONV_LINEAR, ops.ACT_NONE
        C(f0_s, None, *T["proj_net"], 1, 1, 0, 0, 128, 128, LIN, ops.ACT_TANH, st.net0, 0, st.h0_s, 0, None, None)
        C(f0_s, None, *T["proj_inp"], 1, 1, 0, 0, 128, 128, LIN, ops.ACT_RELU, None, 0, st.inp_s, 0, None, None)
        # loop-invariant shares of the four GRU convolutions (bias included), fp32
        st.pre_zr1, st.pre_q1, st.pre_zr2, st.pre_q2 = f32(256), f32(128), f32(256), f32(128)
        bn_zr = _bn256(b, h, w)
        C(st.h0_s, st.inp_s, *T["zr1_fix"], 1, 5, 0, 2, 256, bn_zr, LIN, NONE, st.pre_zr1, 0, None, 0, None, None)
        C(st.inp_s, None, *T["q1_fix"], 1, 5, 0, 2, 128, 128, LIN, NONE, st.pre_q1, 0, None, 0, None, None)
        C(st.inp_s, None, *T["zr2_fix"], 5, 1, 2, 0, 256, bn_zr, LIN, NONE, st.pre_zr2, 0, None, 0, None, None)
        C(st.inp_s, None, *T["q2_fix"], 5, 1, 2, 0, 128, 128, LIN, NONE, st.pre_q2, 0, None, 0, None, None)
        return st

    def _update_block(self, P, st, corr, flow, want_mask):
        """BasicUpdateBlock.forward (reg_refine.py:106-119) as 11 tensor-core convolutions: activations live as fp16 (hi, lo)
        planes, the concatenations are channel offsets / second sources, the GRU gate math is the conv epilogue.
        corr: fp32 correlation volume, or None when it is already in st.corr_s."""
        T, w = P["tc"], P["raw"]
        fd = T["fd"]
        C, L, R = self._conv, ops.CONV_LINEAR, ops.ACT_RELU
        b, h, wd, _ = flow.shape
        dev = flow.device
        bn_zr = bn_fh = _bn256(b, h, wd)
        if corr is not None:
            _OPS.split_planes(corr, st.corr_s, 0)
        C(st.corr_s, None, *T["convc1"], 1, 1, 0, 0, 256, 256, L, R, None, 0, st.cor1_s, 0, None, None)
        C(st.cor1_s, None, *T["convc2"], 3, 3, 1, 1, 192, 96 if bn_zr == 128 else 192, L, R, None, 0, st.cf_s, 0, None, None)
        _OPS.conv7x7_small(flow, None, False, w["refine.encoder.convf1.weight"], w["refine.encoder.convf1.bias"], 1, True,
                           None, None, None, st.flo1_s)        # 7x7 on 1-2 channels: direct fp32 kernel -> fp16 planes
        C(st.flo1_s, None, *T["convf2"], 3, 3, 1, 1, 64, 64, L, R, None, 0, st.cf_s, 192, None, None)
        C(st.cf_s, None, *T["conv"], 3, 3, 1, 1, 128 - fd, 128, L, R, None, 0, st.mfx_s, 0, None, None)
        _OPS.split_planes(flow, st.mfx_s, 128 - fd)                              # mfx = [motion features | flow]
        # SepConvGRU (reg_refine.py:37-52): horizontal 1x5 then vertical 5x1; the invariant input channels come in through `pre`
        Z, Q = ops.CONV_GRU_ZR, ops.CONV_GRU_Q
        kw = dict(gamma=None, beta=None, stride=1, rows=0, win_dst=None, win_geom=None, win_c0=0, win_c1=0, win_streams=0)
        C(st.mfx_s, None, T["zr1_var"], None, 1, 5, 0, 2, 256, bn_zr, Z, 0, st.z, 0, st.rh_s, 0, st.net0, None, pre=st.pre_zr1, **kw)
        C(st.rh_s, st.mfx_s, T["q1_var"], None, 1, 5, 0, 2, 128, 128, Q, 0, st.h1, 0, st.h1_s, 0, st.net0, st.z, pre=st.pre_q1, **kw)
        C(st.h1_s, st.mfx_s, T["zr2_var"], None, 5, 1, 2, 0, 256, bn_zr, Z, 0, st.z, 0, st.rh_s, 0, st.h1, None, pre=st.pre_zr2, **kw)
        C(st.rh_s, st.mfx_s, T["q2_var"], None, 5, 1, 2, 0, 128, 128, Q, 0, st.h2, 0, st.h2_s, 0, st.h1, st.z, pre=st.pre_q2, **kw)
        C(st.h2_s, None, *T["fh1"], 3, 3, 1, 1, 256, bn_fh, L, R, None, 0, st.fh_s, 0, None, None)
        delta = torch.empty((b, h, wd, fd), device=dev)
        C(st.fh_s, None, *T["fh2"], 3, 3, 1, 1, fd, 16, L, ops.ACT_NONE, delta, 0, None, 0, None, None)
        mask = None
        if want_mask and "mask0" in T:
            C(st.h2_s, None, *T["mask0"], 3, 3, 1, 1, 256, bn_fh, L, R, None, 0, st.fh_s, 0, None, None)
            nm = w["refine.mask.2.weight"].shape[0]
            mask = torch.empty((b, h, wd, nm), device=dev)
            C(st.fh_s, None, *T["mask2"], 1, 1, 0, 0, nm, 64, L, ops.ACT_NONE, mask, 0, None, 0, None, None)
        return st.h2, mask, delta

    @staticmethod
    def _refine_feature_planes(rst, g0, g1):
        """fp16 (hi, lo) planes of the correlation features, split once per forward: every iteration reuses them."""
        cached = getattr(rst, "g_planes", None)
        if cached is None or cached[0] is not g0 or cached[1] is not g1:
            planes = []
            for g in (g0, g1):
                gs = torch.empty((2,) + tuple(g.shape), device=g.device, dtype=torch.float16)
                _OPS.split_planes(g, gs, 0)
                planes.append(gs)
            rst.g_planes = (g0, g1, planes[0], planes[1])
        return rst.g_planes[2], rst.g_planes[3]

    def _stage_refine_iter(self, P, rst, g0, g1, flow, task, want_mask, depth=None):
        """One regression-refinement iteration (unimatch.py:272-354): 9x9 correlation volume at the current estimate on the
        pre-transformer features, update block, residual update.  Returns (flow, mask or None)."""
        h, wd = flow.shape[1], flow.shape[2]
        if task == "depth":
            Kr, pr, min_depth, max_depth = depth
            cflow = self._rigid_flow(flow, Kr.float(), pr.float(), h, wd)
        else:
            cflow = flow.contiguous()                                       # disparity handled in-kernel
        with self._section("refine_corr_volume"):
            if _CORR_TC and g0.is_cuda:
                # the volume goes straight into the update block's operand planes (81 of 128 channels).  The op has only a
                # CUDA kernel (TMA + TMEM); CPU tensors, which only the host-logic tests' oracle kernels accept, keep the fp32 op
                g0_s, g1_s = self._refine_feature_planes(rst, g0, g1)
                _OPS.local_corr_volume_planes(g0_s, g1_s, cflow, h, wd, 4, None, rst.corr_s, 0, None)
                corr = None
            else:
                corr = _OPS.local_corr_volume(g0, g1, cflow, h, wd, 4)
        with self._section("refine_update_block"):
            _, mask, delta = self._update_block(P, rst, corr, flow.contiguous(), want_mask)
        if task == "depth":
            flow = (flow - delta).clamp(min=min_depth, max=max_depth)
        else:
            flow = flow + delta
        if task == "stereo":
            flow = flow.clamp(min=0)
        return flow, mask

    def _stage_upsample_learned(self, P, flow2, feat, factor, mult):
        """unimatch.py:81-93 (convex branch): mask = upsampler(cat(flow, feature)) as two tensor-core convolutions
        (3x3 130 -> 256 + ReLU, 1x1 256 -> 9 F^2), then convex upsampling.  flow2: [B,h,w,2]; feat: [B,h,w,128]."""
        U = P["up"]
        b, h, w, _ = feat.shape
        dev = feat.device
        C = self._conv
        src = self._zero_padded("upsampler", (2, b, h, w, 192), dev)                # [feature 0..127 | flow 128..129 | 0]
        _OPS.split_planes(feat.contiguous(), src, 0)
        _OPS.split_planes(flow2.contiguous(), src, 128)
        mid = torch.empty((2, b, h, w, 256), device=dev, dtype=torch.float16)
        C(src, None, *U["c0"], 3, 3, 1, 1, 256, _bn256(b, h, w), ops.CONV_LINEAR, ops.ACT_RELU, None, 0, mid, 0, None, None)
        m = torch.empty((b, h, w, U["nm"]), device=dev)
        C(mid, None, *U["c2"], 1, 1, 0, 0, U["nm"], U["bn2"], ops.CONV_LINEAR, ops.ACT_NONE, m, 0, None, 0, None, None)
        return _OPS.convex_upsample(flow2.contiguous(), m, factor, float(mult))

    @staticmethod
    def _rigid_flow(inv_depth, K, pose, h, w):
        """compute_flow_with_depth_pose(1/inv_depth, K, pose) (geometry.py:99-195) on [B,h,w,1] -> [B,h,w,2]."""
        b = inv_depth.shape[0]
        dev = inv_depth.device
        ys, xs = torch.meshgrid(torch.arange(h, device=dev, dtype=torch.float32),
                                torch.arange(w, device=dev, dtype=torch.float32), indexing="ij")
        grid = torch.stack([xs, ys, torch.ones_like(xs)], dim=0).view(1, 3, -1).expand(b, 3, h * w)
        depth = (1.0 / inv_depth.view(b, 1, h * w))
        pts = torch.inverse(K).bmm(grid) * depth
        pts = torch.bmm(pose[:, :3, :3], pts) + pose[:, :3, -1:]
        proj = torch.bmm(K, pts)
        z = proj[:, 2:3].clamp(min=1e-3)
        uv = proj[:, :2] / z - grid[:, :2]
        return uv.view(b, 2, h, w).permute(0, 2, 3, 1).contiguous()

    # ------------------------------------------------------------------------------------------ forward
    def forward(self, img0, img1, attn_type=None, attn_splits_list=None, corr_radius_list=None, prop_radius_list=None,
                num_reg_refine=1, pred_bidir_flow=False, task="flow", intrinsics=None, pose=None,
                min_depth=1. / 0.5, max_depth=1. / 10, num_depth_candidates=64, depth_from_argmax=False,
                pred_bidir_depth=False, **kwargs):
        if self.training:
            raise NotImplementedError("unimatch_b200.UniMatch is inference-only; call .eval()")
        if pred_bidir_flow:
            assert task == "flow"
        if task == "depth":
            assert self.num_scales == 1
            assert len(attn_splits_list) == len(prop_radius_list) == self.num_scales == 1
        else:
            assert len(attn_splits_list) == len(corr_radius_list) == len(prop_radius_list) == self.num_scales
        # no device check here: the unimatch_sm100 ops are registered for CUDA only, so CPU tensors fail loudly
        # in the dispatcher (there is no CPU path)
        with torch.no_grad():
            return self._forward(img0, img1, attn_type, attn_splits_list, corr_radius_list, prop_radius_list,
                                 num_reg_refine, pred_bidir_flow, task, intrinsics, pose, min_depth, max_depth,
                                 num_depth_candidates, depth_from_argmax, pred_bidir_depth)

    def _forward(self, img0, img1, attn_type, attn_splits_list, corr_radius_list, prop_radius_list, num_reg_refine,
                 pred_bidir_flow, task, intrinsics, pose, min_depth, max_depth, num_depth_candidates,
                 depth_from_argmax, pred_bidir_depth):
        P = self._prepared()
        B = img0.shape[0]
        with self._section("backbone"):                                           # [2B,h,w,128] low -> high res
            feats = self._stage_backbone(P, img0.float().contiguous(), img1.float().contiguous(), task == "flow")

        flow = None            # [Bp, h, w, fd] channel-last
        preds = []
        for s in range(self.num_scales):
            f = feats[s]
            _, h, wd, c = f.shape
            f0, f1 = f[:B], f[B:]
            if pred_bidir_flow and s > 0:                                         # unimatch.py:139-141
                f0, f1 = torch.cat((f0, f1), dim=0), torch.cat((f1, f0), dim=0)
            f0_ori, f1_ori = f0, f1
            Bp = f0.shape[0]
            up = self.upsample_factor * (2 ** (self.num_scales - 1 - s))
            Ks = None
            if task == "depth":
                Ks = intrinsics.clone().float()
                Ks[:, :2] = Ks[:, :2] / up
            if s > 0:
                flow = _OPS.upsample2x(flow.contiguous(), 2.0)                    # unimatch.py:154
            splits = attn_splits_list[s]
            prop_r = prop_radius_list[s]
            tok = self._stage_features(f0, f1, flow, h, wd, splits)
            with self._section("transformer_s%d" % s):
                tok, tok_s = self._stage_transformer(P, tok, h, wd, attn_type, splits, "s%d" % s)   # [2Bp, L, 128]

            # ---- correlation + softmax (unimatch.py:186-216) ----
            with self._section("correlation_s%d" % s):
                dargs = (Ks, pose, min_depth, max_depth, num_depth_candidates, depth_from_argmax, pred_bidir_depth) \
                    if task == "depth" else None
                pred = self._stage_correlation(tok, Bp, h, wd, task, None if task == "depth" else corr_radius_list[s],
                                               pred_bidir_flow, dargs)
            flow = flow + pred if flow is not None else pred
            if task == "stereo":
                flow = flow.clamp(min=0)

            # ---- self-attention propagation (unimatch.py:230-237, attention.py:184-253) ----
            bidir0 = (pred_bidir_flow or pred_bidir_depth) and s == 0
            nb = 2 * Bp if bidir0 else Bp                                         # bidirectional: cat(feature0, feature1)
            with self._section("propagation_s%d" % s):
                flow = self._stage_propagation(P, tok_s, flow, nb, h, wd, prop_r)
            if s != self.num_scales - 1:
                continue

            feat0 = tok[:nb].reshape(nb, h, wd, c)                                # post-transformer feature0
            if not self.reg_refine:                                               # unimatch.py:246-264
                zeros = torch.zeros_like(flow)
                if task == "stereo":
                    out = -self._stage_upsample_learned(P, torch.cat((-flow, zeros), -1), feat0, self.upsample_factor,
                                                        self.upsample_factor)[:, :1]
                elif task == "depth":
                    out = self._stage_upsample_learned(P, torch.cat((flow, zeros), -1), feat0, self.upsample_factor,
                                                       1).clamp(min=min_depth, max=max_depth)[:, :1]
                else:
                    out = self._stage_upsample_learned(P, flow, feat0, self.upsample_factor, self.upsample_factor)
                preds.append(out)
                continue

            # ---- regression refinement (unimatch.py:272-354) ----
            assert num_reg_refine > 0
            g0, g1 = f0_ori.contiguous(), f1_ori.contiguous()
            drefine = None
            if task == "depth":
                Kr, pr = Ks, pose
                if pred_bidir_depth:
                    Kr = Ks.repeat(2, 1, 1)
                    pr = torch.cat((pose, torch.inverse(pose)), dim=0).float()
                    g0, g1 = torch.cat((g0, g1), dim=0), torch.cat((g1, g0), dim=0)
                drefine = (Kr, pr, min_depth, max_depth)
            rst = self._stage_refine_setup(P, feat0.contiguous(), nb, h, wd)
            for it in range(num_reg_refine):
                last = it == num_reg_refine - 1
                flow, mask = self._stage_refine_iter(P, rst, g0, g1, flow, task, last, drefine)
                if last:
                    if task == "depth":
                        out = self._stage_upsample_learned(P, torch.cat((flow, torch.zeros_like(flow)), -1), feat0,
                                                           self.upsample_factor, 1).clamp(min=min_depth, max=max_depth)[:, :1]
                    else:
                        out = _OPS.convex_upsample(flow.contiguous(), mask, self.upsample_factor,
                                                   float(self.upsample_factor))
                    preds.append(out)

        if task == "stereo":
            preds = [p.squeeze(1) for p in preds]
        if task == "depth":
            preds = [1.0 / p.squeeze(1) for p in preds]
        return {"flow_preds": preds}
