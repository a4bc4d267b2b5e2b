"""Op-level parity on the GPU: every `torch.ops.unimatch_sm100.*` kernel (called through the C ABI) against the
oracle-backed reference of the same name in tests/refops.py, on identical seeded inputs.
Tolerances (fp32 path): max |diff| <= TOL * max(1, max |ref|); TOL stated per test."""
import pytest
import torch

import refops
from unimatch_b200 import ops

pytestmark = pytest.mark.gpu
OPS = torch.ops.unimatch_sm100
C = 128


def g(seed):
    return torch.Generator().manual_seed(seed)


def close(got, ref, tol):
    got = got.detach().float().cpu()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    assert torch.isfinite(got).all()
    err = (got - ref).abs().max().item()
    lim = tol * max(1.0, ref.abs().max().item())
    assert err <= lim, "max|diff| %.3e > %.3e" % (err, lim)


ATTN_CASES = [
    # n, h, w, kh, kw, shift, kv_shift
    (2, 6, 8, 1, 1, False, 0),          # full 2-D
    (2, 12, 16, 2, 2, False, 1),        # swin windows, cross pairing
    (2, 12, 16, 2, 2, True, 1),         # shifted + region mask
    (2, 16, 24, 4, 4, True, 0),
    (2, 30, 52, 2, 2, True, 1),         # Lw = 390: ragged vs the 64-wide tiles
    (4, 15, 26, 1, 1, False, 2),        # Lw = 390, full
    (2, 5, 24, 5, 4, True, 1),          # 1-D windows along rows, shifted
    (2, 5, 24, 5, 4, False, 0),
    (2, 6, 40, 6, 1, False, 1),         # full 1-D rows
    (2, 8, 70, 1, 1, False, 0),         # L = 560, several key tiles
]


@pytest.mark.parametrize("n,h,w,kh,kw,shift,kvs", ATTN_CASES)
def test_window_attention(n, h, w, kh, kw, shift, kvs):
    gen = g(100 + h * w + kh)
    L = h * w
    qkv = torch.randn((n, L, 3 * C), generator=gen) * 1.5        # strided views, like the fused projection output
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    wh, ww = h // kh, w // kw
    sh = (wh // 2 if kh != h else 0) if shift else 0
    sw = ww // 2 if shift else 0
    mask = ops.MASK_SWIN if shift else ops.MASK_NONE
    ref = refops.window_attention(q, k, v, kvs, h, w, kh, kw, sh, sw, mask)
    d = qkv.cuda()
    got = OPS.window_attention(d[..., :C], d[..., C:2 * C], d[..., 2 * C:], kvs, h, w, kh, kw, sh, sw, mask)
    close(got, ref, 2e-5)


EXP_CASES = [
    # n_total, n_streams, kv_shift, h, w, vdim, value_mode, post, kh, kw, mask
    (4, 2, 2, 7, 9, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN, 1, 1, ops.MASK_NONE),      # global corr
    (4, 4, 2, 7, 9, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN, 1, 1, ops.MASK_NONE),      # bidirectional
    (2, 1, 1, 12, 30, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN, 1, 1, ops.MASK_NONE),    # L = 360
    (4, 2, 2, 5, 14, 1, ops.VALUE_XCOORD, ops.POST_OWN_MINUS, 5, 1, ops.MASK_CAUSAL),   # stereo rows
    (2, 1, 1, 3, 100, 1, ops.VALUE_XCOORD, ops.POST_OWN_MINUS, 3, 1, ops.MASK_CAUSAL),  # W = 100 > one key tile
    (2, 2, 0, 7, 9, 2, ops.VALUE_TENSOR, ops.POST_NONE, 1, 1, ops.MASK_NONE),           # global propagation
    (3, 3, 0, 9, 11, 1, ops.VALUE_TENSOR, ops.POST_NONE, 1, 1, ops.MASK_NONE),
    (2, 2, 0, 12, 30, 2, ops.VALUE_TENSOR, ops.POST_NONE, 1, 1, ops.MASK_NONE),         # L = 360: tensor-core path
    (2, 2, 0, 16, 24, 1, ops.VALUE_TENSOR, ops.POST_NONE, 1, 1, ops.MASK_NONE),         # L = 384 = 3 full tiles
    (4, 4, 2, 12, 16, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN, 1, 1, ops.MASK_NONE),    # bidirectional, L = 192
]


@pytest.mark.parametrize("nt,ns,kvs,h,w,vdim,vm,post,kh,kw,mask", EXP_CASES)
def test_softmax_expectation(nt, ns, kvs, h, w, vdim, vm, post, kh, kw, mask):
    gen = g(200 + h * w + vdim)
    L = h * w
    q = torch.randn((nt, L, C), generator=gen) * 1.5
    k = torch.randn((nt, L, C), generator=gen) * 1.5
    vals = torch.randn((nt, L, vdim), generator=gen) * 3 if vm == ops.VALUE_TENSOR else None
    ref = refops.softmax_expectation(q, k, vals, ns, kvs, vdim, vm, post, h, w, kh, kw, mask)
    got = OPS.softmax_expectation(q.cuda(), k.cuda(), None if vals is None else vals.cuda(), ns, kvs, vdim, vm, post,
                                  h, w, kh, kw, mask)
    close(got, ref, 2e-5)


def feats(seed, b, h, w, scale=1.5):
    gen = g(seed)
    return torch.randn((b, h, w, C), generator=gen) * scale, torch.randn((b, h, w, C), generator=gen) * scale, gen


@pytest.mark.parametrize("b,h,w,ry,rx,stereo", [(2, 11, 13, 4, 4, False), (1, 20, 33, 4, 4, False),
                                                (2, 5, 14, 0, 4, True), (1, 9, 40, 0, 4, True)])
def test_local_corr_softmax(b, h, w, ry, rx, stereo):
    f0, f1, _ = feats(300 + h, b, h, w)
    ref = refops.local_corr_softmax(f0, f1, h, w, ry, rx, stereo)
    got = OPS.local_corr_softmax(f0.cuda(), f1.cuda(), h, w, ry, rx, stereo)
    close(got, ref, 2e-5)


@pytest.mark.parametrize("b,h,w,fd,mag", [(2, 11, 13, 2, 3.0), (1, 20, 33, 2, 12.0), (2, 9, 17, 1, 4.0),
                                          (1, 8, 8, 2, 0.0)])
def test_local_corr_volume(b, h, w, fd, mag):
    f0, f1, gen = feats(400 + h, b, h, w)
    flow = torch.randn((b, h, w, fd), generator=gen) * mag          # large flows push windows out of the image
    ref = refops.local_corr_volume(f0, f1, flow, h, w, 4)
    got = OPS.local_corr_volume(f0.cuda(), f1.cuda(), flow.cuda(), h, w, 4)
    close(got, ref, 3e-5)


@pytest.mark.parametrize("b,h,w,fd,mag", [(2, 9, 12, 2, 4.0), (1, 16, 20, 2, 30.0), (2, 9, 12, 1, 5.0)])
def test_flow_warp(b, h, w, fd, mag):
    _, f1, gen = feats(500 + h, b, h, w)
    flow = torch.randn((b, h, w, fd), generator=gen) * mag
    ref = refops.flow_warp(f1, flow, h, w)
    got = OPS.flow_warp(f1.cuda(), flow.cuda(), h, w)
    close(got, ref, 1e-5)


def test_flow_warp_zero_flow_is_identity():
    _, f1, _ = feats(510, 2, 10, 14)
    got = OPS.flow_warp(f1.cuda(), torch.zeros(2, 10, 14, 2).cuda(), 10, 14)
    close(got, f1, 1e-6)


@pytest.mark.parametrize("b,h,w,fd", [(2, 7, 9, 2), (2, 7, 9, 1), (1, 12, 30, 2)])
def test_propagate_local(b, h, w, fd):
    gen = g(600 + w)
    q = torch.randn((b, h * w, C), generator=gen) * 1.5
    k = torch.randn((b, h * w, C), generator=gen) * 1.5
    flow = torch.randn((b, h, w, fd), generator=gen) * 3
    ref = refops.propagate_local(q, k, flow, h, w, 1)
    got = OPS.propagate_local(q.cuda(), k.cuda(), flow.cuda(), h, w, 1)
    close(got, ref, 2e-5)


@pytest.mark.parametrize("argmax", [False, True])
def test_depth_corr_softmax(argmax):
    b, h, w, d = 2, 8, 10, 16
    f0, f1, _ = feats(700, b, h, w, 1.0)
    K = torch.tensor([[0.9 * w, 0.0, w / 2.0], [0.0, 0.9 * w, h / 2.0], [0.0, 0.0, 1.0]]).view(1, 3, 3).repeat(b, 1, 1)
    pose = torch.eye(4).view(1, 4, 4).repeat(b, 1, 1)
    pose[:, 0, 3] = 0.1
    pose[:, 2, 3] = 0.02
    cand = torch.linspace(0.1, 2.0, d)
    Kinv = torch.inverse(K).contiguous()
    ref = refops.depth_corr_softmax(f0, f1, K, Kinv, pose, cand, h, w, argmax)
    got = OPS.depth_corr_softmax(f0.cuda(), f1.cuda(), K.cuda(), Kinv.cuda(), pose.cuda(), cand.cuda(), h, w, argmax)
    close(got, ref, 2e-5)


def test_add_position():
    from unimatch_b200.unimatch import _sine_table
    x = torch.randn((3, 8, 12, C), generator=g(800))
    table = _sine_table(4, 6)
    close(OPS.add_position(x.cuda(), table.cuda(), 8, 12), refops.add_position(x, table, 8, 12), 1e-6)


def test_sine_table_is_the_reference_encoding():
    from oracle import unimatch_oracle as O
    from unimatch_b200.unimatch import _sine_table
    ref = O.sine_position(torch.zeros(1, C, 5, 7))[0].permute(1, 2, 0)
    assert (ref - _sine_table(5, 7)).abs().max().item() <= 1e-6


@pytest.mark.parametrize("with_res", [False, True])
def test_layernorm_residual(with_res):
    gen = g(900)
    x = torch.randn((2, 37, C), generator=gen) * 3 + 0.5
    res = torch.randn((2, 37, C), generator=gen) if with_res else None
    gamma, beta = torch.randn(C, generator=gen), torch.randn(C, generator=gen)
    ref = refops.layernorm_residual(x, res, gamma, beta)
    got = OPS.layernorm_residual(x.cuda(), None if res is None else res.cuda(), gamma.cuda(), beta.cuda())
    close(got, ref, 1e-5)


@pytest.mark.parametrize("fd,factor,mult", [(2, 4, 4.0), (2, 8, 8.0), (2, 8, 1.0)])
def test_convex_upsample(fd, factor, mult):
    gen = g(1000 + factor)
    flow = torch.randn((2, 6, 7, fd), generator=gen) * 2
    mask = torch.randn((2, 6, 7, 9 * factor * factor), generator=gen) * 3
    close(OPS.convex_upsample(flow.cuda(), mask.cuda(), factor, mult), refops.convex_upsample(flow, mask, factor, mult), 1e-5)


@pytest.mark.parametrize("fd", [1, 2])
def test_upsample2x(fd):
    flow = torch.randn((2, 7, 9, fd), generator=g(1100)) * 5
    close(OPS.upsample2x(flow.cuda(), 2.0), refops.upsample2x(flow, 2.0), 1e-5)


def test_gru_gates():
    gen = g(1200)
    zr = torch.randn((2, 5, 6, 256), generator=gen) * 2
    q = torch.randn((2, 5, 6, C), generator=gen) * 2
    h = torch.tanh(torch.randn((2, 5, 6, C), generator=gen))
    d = zr.cuda()
    close(OPS.gru_rh(d[..., 128:], h.cuda()), refops.gru_rh(zr[..., 128:], h), 1e-5)
    close(OPS.gru_update(d[..., :128], q.cuda(), h.cuda()), refops.gru_update(zr[..., :128], q, h), 1e-5)


CONV_CASES = [
    # name, cins, cout, kh, kw, bn, mode, act, (h, w)
    ("convc1_1x1", [81], 256, 1, 1, 128, "lin", ops.ACT_RELU, (16, 32)),
    ("convc2_3x3", [256], 192, 3, 3, 64, "lin", ops.ACT_RELU, (20, 33)),
    ("conv_3x3_126", [256], 126, 3, 3, 128, "lin", ops.ACT_RELU, (16, 16)),
    ("gru_zr_1x5", [128, 256], 256, 1, 5, 128, "zr", 0, (12, 40)),
    ("gru_q_5x1", [128, 256], 128, 5, 1, 128, "q", 0, (24, 16)),
    ("flow_head2_3x3", [256], 2, 3, 3, 16, "lin", ops.ACT_NONE, (9, 21)),
    ("mask2_1x1", [256], 144, 1, 1, 64, "lin", ops.ACT_NONE, (8, 16)),
    ("proj_tanh", [128], 128, 1, 1, 128, "lin", ops.ACT_TANH, (8, 16)),
    ("linear_ln_residual", [128], 128, 1, 1, 128, "ln", 0, (40, 16)),            # token rows as a [rows/16, 16] grid
    ("ffn1_two_sources_gelu", [128, 128], 1024, 1, 1, 128, "lin", ops.ACT_GELU, (24, 16)),
    ("ffn2_k1024_ln", [1024], 128, 1, 1, 128, "ln", 0, (24, 16)),
    ("many_tiles_persistent", [128], 640, 1, 1, 128, "lin", ops.ACT_NONE, (400, 16)),   # 250 tiles > 148 SMs
    # wide tiles (BN = 192 / 256: two 96 KB stages, one TMEM accumulator buffer)
    ("convc2_3x3_bn192", [256], 192, 3, 3, 192, "lin", ops.ACT_RELU, (20, 33)),
    ("gru_zr_1x5_bn256", [128, 256], 256, 1, 5, 256, "zr", 0, (12, 40)),
    ("flow_head1_3x3_bn256", [128], 256, 3, 3, 256, "lin", ops.ACT_RELU, (24, 40)),
    ("convc1_1x1_bn256", [81], 256, 1, 1, 256, "lin", ops.ACT_RELU, (16, 32)),
    ("wide_many_tiles", [128], 256, 3, 3, 256, "lin", ops.ACT_RELU, (160, 128)),        # 320 tiles: several per CTA
    ("ffn1_two_sources_gelu_bn256", [128, 128], 1024, 1, 1, 256, "lin", ops.ACT_GELU, (24, 16)),
    # CTA-pair kernels (cta_group::2; taken for long-K launches with an even number of pixel tiles -- most cases above with
    # batch 2 already are): LayerNorm epilogue on a pair, several tiles per pair with G = 2 / G = 4, an odd tile count per
    # CTA pair on the last round (76 pair tiles on 74 clusters)
    ("ffn2_k1024_ln_pair", [1024], 128, 1, 1, 128, "ln", 0, (32, 16)),
    ("ffn2_k1024_ln_pair_many", [1024], 128, 1, 1, 128, "ln", 0, (2432, 16)),
    ("pair_many_tiles_bn128", [256], 128, 3, 3, 128, "lin", ops.ACT_RELU, (160, 128)),
    ("pair_many_tiles_bn64", [128], 64, 3, 3, 64, "lin", ops.ACT_NONE, (152, 64)),
    ("gru_q_5x1_pair_many", [128, 256], 128, 5, 1, 128, "q", 0, (152, 64)),
    ("convc2_3x3_bn96_pair", [256], 192, 3, 3, 96, "lin", ops.ACT_RELU, (152, 64)),   # 192 channels as 2 x 96, 76 pair tiles
]


@pytest.mark.parametrize("name,cins,cout,kh,kw,bn,mode,act,hw", CONV_CASES)
def test_conv2d_tc(name, cins, cout, kh, kw, bn, mode, act, hw):
    """Tensor-core implicit-GEMM convolution vs the fp32 convolution of the same (hi+lo) operands."""
    h, w = hw
    b = 2
    gen = g(2000 + cout + kh)
    cin = sum(cins)
    wt = torch.randn((cout, cin, kh, kw), generator=gen) * (2.0 / (cin * kh * kw)) ** 0.5
    bias = torch.randn(cout, generator=gen) * 0.1
    cout_p = (cout + bn - 1) // bn * bn
    wp = ops.prep_conv_weight(wt, cins, cout_p)
    xs = [torch.randn((b, h, w, c), generator=gen) for c in cins]
    hh = torch.tanh(torch.randn((b, h, w, 128), generator=gen))
    zz = torch.sigmoid(torch.randn((b, h, w, 128), generator=gen))
    m = {"lin": ops.CONV_LINEAR, "zr": ops.CONV_GRU_ZR, "q": ops.CONV_GRU_Q, "ln": ops.CONV_LN}[mode]
    gamma, beta = torch.randn(128, generator=gen), torch.randn(128, generator=gen)
    if mode == "ln":
        b = 1
        xs = [x[:1] for x in xs]
        hh, zz = hh[:1], zz[:1]

    def run(dev, conv_fn, split_fn):
        srcs = []
        for x, c in zip(xs, cins):
            buf = torch.zeros((2, b, h, w, (c + 63) // 64 * 64), dtype=torch.float16, device=dev)
            split_fn(x.to(dev), buf, 0)
            srcs.append(buf)
        out_f = torch.zeros((b, h, w, (cout + 7) // 4 * 4), device=dev)     # written at channel offset 4 (offset stores)
        out_s = torch.zeros((2, b, h, w, 192 if cout <= 128 else cout + 64), dtype=torch.float16, device=dev)
        conv_fn(srcs[0], srcs[1] if len(srcs) > 1 else None, wp.to(dev), None if mode == "ln" else bias.to(dev), kh, kw,
                kh // 2, kw // 2, cout, bn, m, act, out_f, 4 if mode != "zr" else 0, out_s, 64,
                hh.to(dev) if mode != "lin" else None, zz.to(dev) if mode == "q" else None,
                gamma.to(dev) if mode == "ln" else None, beta.to(dev) if mode == "ln" else None)
        return out_f.cpu(), (out_s[0].float() + out_s[1].float()).cpu()

    ref_f, ref_s = run("cpu", refops.conv2d_tc, refops.split_planes)
    got_f, got_s = run("cuda", OPS.conv2d_tc, OPS.split_planes)
    close(got_f, ref_f, 2e-5)
    close(got_s, ref_s, 2e-5)
    # and the hi+lo operands themselves reproduce the fp32 convolution of the unsplit inputs
    y = torch.nn.functional.conv2d(torch.cat(xs, -1).permute(0, 3, 1, 2), wt, bias, padding=(kh // 2, kw // 2))
    if mode == "lin" and act == ops.ACT_NONE:
        close(got_f[..., 4:4 + cout], y.permute(0, 2, 3, 1).contiguous(), 2e-5)


@pytest.mark.parametrize("rows,hidden,outs", [(256, 128, "both"), (512, 1024, "both"), (256 * 77, 1024, "both"),
                                              (256 * 150, 256, "split"), (1024, 1024, "f32")])
def test_ffn_tc(rows, hidden, outs):
    """Fused FFN (CTA-pair kernel, hidden activation in tensor memory) vs the two GEMM launches it replaces, stated on CPU
    (tests/refops.py): one chunk, the module's 8 chunks, more tile pairs than clusters (77 and 150 on 74)."""
    gen = g(7000 + rows % 997 + hidden)
    w1 = torch.randn((hidden, 256, 1, 1), generator=gen) * (2.0 / 256) ** 0.5
    w2 = torch.randn((128, hidden, 1, 1), generator=gen) * (1.0 / hidden) ** 0.5
    w1p, w2p = ops.prep_conv_weight(w1, [128, 128], hidden), ops.prep_conv_weight(w2, [hidden], 128)
    pad = 32                                                               # plane buffers longer than `rows`
    xs = [torch.randn((rows, 128), generator=gen) for _ in range(2)]
    res = torch.randn((rows + pad, 128), generator=gen)
    gamma, beta = torch.randn(128, generator=gen), torch.randn(128, generator=gen)

    def run(dev, ffn_fn, split_fn):
        srcs = []
        for x in xs:
            buf = torch.zeros((2, rows + pad, 128), dtype=torch.float16, device=dev)
            split_fn(x.to(dev), buf, 0)
            srcs.append(buf)
        out_f = torch.zeros((rows + pad, 128), device=dev) if outs != "split" else None
        out_s = torch.zeros((2, rows + pad, 128), dtype=torch.float16, device=dev) if outs != "f32" else None
        ffn_fn(srcs[0], srcs[1], w1p.to(dev), w2p.to(dev), res.to(dev), gamma.to(dev), beta.to(dev), out_f, out_s, rows)
        return (out_f.cpu() if out_f is not None else None,
                (out_s[0].float() + out_s[1].float()).cpu() if out_s is not None else None)

    ref_f, ref_s = run("cpu", refops.ffn_tc, refops.split_planes)
    for rep in range(2):                                                   # twice: barrier phases / TMEM state carry nothing over
        got_f, got_s = run("cuda", OPS.ffn_tc, OPS.split_planes)
        if ref_f is not None:
            close(got_f, ref_f, 3e-5)
            assert got_f[rows:].abs().max().item() == 0.0                  # rows beyond `rows` untouched
        if ref_s is not None:
            close(got_s, ref_s, 3e-5)


@pytest.mark.parametrize("outs", ["f32", "split"])
@pytest.mark.parametrize("cout,act", [(640, ops.ACT_NONE), (1024, ops.ACT_GELU), (128, ops.ACT_RELU)])
def test_conv2d_tc_single_output_many_tiles(cout, act, outs):
    """One output kind only (the way the module calls the Linear layers / encoder convolutions): the epilogue then
    double-buffers its staging tiles across chunks and tiles, so a persistent CTA with many tiles must never overwrite
    a staging buffer a bulk store is still reading.  ~6-45 tiles per CTA; repeated to give a race a chance to show."""
    rows_grid, b = (1200, 16), 1                                            # 150 pixel tiles x cout/128 channel tiles
    gen = g(4100 + cout)
    wt = torch.randn((cout, 128, 1, 1), generator=gen) * (2.0 / 128) ** 0.5
    bias = torch.randn(cout, generator=gen) * 0.1
    wp = ops.prep_conv_weight(wt, [128], cout)
    x = torch.randn((b, rows_grid[0], rows_grid[1], 128), generator=gen)

    def run(dev, conv_fn, split_fn):
        src = torch.zeros((2, b, *rows_grid, 128), dtype=torch.float16, device=dev)
        split_fn(x.to(dev), src, 0)
        out_f = torch.zeros((b, *rows_grid, cout), device=dev) if outs == "f32" else None
        out_s = torch.zeros((2, b, *rows_grid, cout), dtype=torch.float16, device=dev) if outs == "split" else None
        res = []
        for _ in range(1 if dev == "cpu" else 4):
            conv_fn(src, None, wp.to(dev), bias.to(dev), 1, 1, 0, 0, cout, 128, ops.CONV_LINEAR, act, out_f, 0, out_s, 0, None, None)
            res.append(out_f.cpu().clone() if outs == "f32" else (out_s[0].float() + out_s[1].float()).cpu())
        return res

    ref = run("cpu", refops.conv2d_tc, refops.split_planes)[0]
    for got in run("cuda", OPS.conv2d_tc, OPS.split_planes):
        close(got, ref, 2e-5)


@pytest.mark.parametrize("cin,cout,k,stride,hw", [(64, 96, 3, 2, (32, 48)), (64, 96, 1, 2, (32, 48)), (128, 128, 3, 2, (30, 52)),
                                                   (96, 128, 3, 1, (20, 33)), (64, 64, 3, 1, (24, 32))])
def test_conv2d_tc_backbone_shapes(cin, cout, k, stride, hw):
    """Strided (TMA elementStrides) and odd-channel convolutions of the CNN encoder vs the fp32 convolution."""
    h, w = hw
    b = 2
    gen = g(3000 + cin + cout + k + stride)
    wt = torch.randn((cout, cin, k, k), generator=gen) * (2.0 / (cin * k * k)) ** 0.5
    bias = torch.randn(cout, generator=gen) * 0.1
    bn = 128 if cout > 64 else 64
    wp = ops.prep_conv_weight(wt, [cin], (cout + bn - 1) // bn * bn)
    x = torch.randn((b, h, w, cin), generator=gen)
    cp = (cin + 63) // 64 * 64
    ho, wo = (h + 2 * (k // 2) - k) // stride + 1, (w + 2 * (k // 2) - k) // stride + 1

    def run(dev, conv_fn, split_fn):
        buf = torch.zeros((2, b, h, w, cp), dtype=torch.float16, device=dev)
        split_fn(x.to(dev), buf, 0)
        out = torch.zeros((b, ho, wo, cout), device=dev)
        conv_fn(buf, None, wp.to(dev), bias.to(dev), k, k, k // 2, k // 2, cout, bn, ops.CONV_LINEAR, ops.ACT_NONE, out, 0,
                None, 0, None, None, None, None, stride)
        return out.cpu()

    ref = run("cpu", refops.conv2d_tc, refops.split_planes)
    got = run("cuda", OPS.conv2d_tc, OPS.split_planes)
    close(got, ref, 2e-5)
    y = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2), wt, bias, stride=stride, padding=k // 2).permute(0, 2, 3, 1)
    close(got, y.contiguous(), 2e-5)


@pytest.mark.parametrize("hw", [(40, 56), (200, 330)])     # the larger one: 312 tiles > 2 CTAs x 148 SMs (persistent loop)
def test_conv7x7_stem_with_folded_normalisation(hw):
    gen = g(3200)
    H, W = hw
    img0 = torch.rand((2, 3, H, W), generator=gen) * 255
    img1 = torch.rand((2, 3, H, W), generator=gen) * 255
    wt = torch.randn((64, 3, 7, 7), generator=gen) * 0.1
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    scale = [1.0 / (255.0 * s_) for s_ in std]
    shift = [-m_ / s_ for m_, s_ in zip(mean, std)]
    ref = torch.zeros((4, H // 2, W // 2, 64))
    refops.conv7x7_small(img0, img1, True, wt, None, 2, False, scale, shift, ref, None)
    out = torch.zeros((4, H // 2, W // 2, 64)).cuda()
    OPS.conv7x7_small(img0.cuda(), img1.cuda(), True, wt.cuda(), None, 2, False, scale, shift, out, None)
    close(out, ref, 1e-5)
    # and against the reference's own two-step form: normalize_img then conv
    x = torch.cat((img0, img1), 0)
    xn = (x / 255.0 - torch.tensor(mean).view(1, 3, 1, 1)) / torch.tensor(std).view(1, 3, 1, 1)
    close(out, torch.nn.functional.conv2d(xn, wt, None, stride=2, padding=3).permute(0, 2, 3, 1).contiguous(), 2e-5)


@pytest.mark.parametrize("fd", [1, 2])
def test_conv7x7_flow_encoder(fd):
    gen = g(3300 + fd)
    flow = torch.randn((2, 19, 27, fd), generator=gen) * 3
    wt = torch.randn((128, fd, 7, 7), generator=gen) * 0.1
    bias = torch.randn(128, generator=gen) * 0.1
    ref_f = torch.zeros((2, 19, 27, 128))
    ref_s = torch.zeros((2, 2, 19, 27, 128), dtype=torch.float16)
    refops.conv7x7_small(flow, None, False, wt, bias, 1, True, None, None, ref_f, ref_s)
    out_f = torch.zeros((2, 19, 27, 128)).cuda()
    out_s = torch.zeros((2, 2, 19, 27, 128), dtype=torch.float16).cuda()
    OPS.conv7x7_small(flow.cuda(), None, False, wt.cuda(), bias.cuda(), 1, True, None, None, out_f, out_s)
    close(out_f, ref_f, 1e-5)
    close(out_s[0].float() + out_s[1].float(), ref_s[0].float() + ref_s[1].float(), 1e-5)


@pytest.mark.parametrize("c", [64, 96, 128])
def test_instance_norm(c):
    gen = g(3100 + c)
    a = torch.randn((3, 20, 28, c), generator=gen) * 2 + 0.7
    res = torch.randn((3, 20, 28, c), generator=gen)
    st_ref = refops.instance_norm_stats(a)
    st = OPS.instance_norm_stats(a.cuda())
    close(st, st_ref, 1e-5)
    # against torch's own instance_norm
    ref = torch.relu(torch.relu(torch.nn.functional.instance_norm(a.permute(0, 3, 1, 2))).permute(0, 2, 3, 1) + res)
    cp = (c + 63) // 64 * 64
    out = torch.zeros((3, 20, 28, c)).cuda()
    pl = torch.zeros((2, 3, 20, 28, cp), dtype=torch.float16).cuda()
    OPS.instance_norm_apply(a.cuda(), st, True, res.cuda(), None, True, out, pl, 0)
    close(out, ref, 1e-5)
    close((pl[0].float() + pl[1].float())[..., :c], ref, 1e-5)
    # normalised residual branch (downsample path)
    st_r = OPS.instance_norm_stats(res.cuda())
    ref2 = torch.relu(torch.relu(torch.nn.functional.instance_norm(a.permute(0, 3, 1, 2))) +
                      torch.nn.functional.instance_norm(res.permute(0, 3, 1, 2))).permute(0, 2, 3, 1)
    OPS.instance_norm_apply(a.cuda(), st, True, res.cuda(), st_r, True, out, None, 0)
    close(out, ref2.contiguous(), 1e-5)


def test_cpu_tensors_are_rejected():
    refops.unregister_cpu_kernels()         # a CPU test earlier in the same session may have installed them
    with pytest.raises((NotImplementedError, RuntimeError)):
        OPS.upsample2x(torch.zeros(1, 2, 2, 2), 2.0)


# ---- size-independent properties at BASELINE shapes (480x832 -> 60x104 and 120x208 feature maps) ------------
def test_attention_of_constant_values_is_constant_fullsize():
    n, h, w = 2, 60, 104
    gen = g(1300)
    q = (torch.randn((n, h * w, C), generator=gen) * 2).cuda()
    k = (torch.randn((n, h * w, C), generator=gen) * 2).cuda()
    v = torch.ones((n, h * w, C)).cuda() * 0.75
    out = OPS.window_attention(q, k, v, 1, h, w, 2, 2, 15, 26, ops.MASK_SWIN)
    # tensor-core fp32 accumulation truncates (round-toward-zero) at each of the ~300 accumulate steps of a
    # 1560-key window: a one-sided bias of up to ~2e-5 relative on an all-positive sum (measured 1.9e-5)
    assert (out - 0.75).abs().max().item() <= 4e-5


def test_global_corr_peaked_match_recovers_translation_fullsize():
    """Keys = queries translated by (dx, dy) with strongly peaked logits -> flow == (dx, dy) away from the border."""
    h, w, dx, dy = 60, 104, 3, -2
    f = torch.randn((1, h, w, C), generator=g(1400)) * 4
    f1 = torch.roll(f, shifts=(dy, dx), dims=(1, 2))
    tok = torch.cat((f, f1), 0).view(2, h * w, C).cuda()
    flow = OPS.softmax_expectation(tok, tok, None, 1, 1, 2, ops.VALUE_COORDS, ops.POST_MINUS_OWN, h, w, 1, 1,
                                   ops.MASK_NONE).view(h, w, 2).cpu()
    inner = flow[4:-4, 4:-4]
    assert (inner[..., 0] - dx).abs().max().item() < 1e-3 and (inner[..., 1] - dy).abs().max().item() < 1e-3


def test_local_corr_volume_zero_flow_equals_shifted_dots_fullsize():
    b, h, w = 1, 120, 208
    f0, f1, _ = feats(1500, b, h, w, 1.0)
    d0, d1 = f0.cuda(), f1.cuda()
    got = OPS.local_corr_volume(d0, d1, torch.zeros(b, h, w, 2).cuda(), h, w, 4)
    pad = torch.nn.functional.pad(d1, (0, 0, 4, 4, 4, 4))
    for k in (0, 8, 40, 44, 80):
        iy, ix = k // 9, k % 9
        ref = (d0 * pad[:, iy:iy + h, ix:ix + w]).sum(-1) / (C ** 0.5)
        assert (got[..., k] - ref).abs().max().item() <= 1e-4


# ---- the tensor-core attention at the BASELINE window shapes, against the ORACLE (reference attention.py:45-104) ---------
FULL_ATTN_CASES = [
    # n, h, w, K, shifted, kv_shift          window length          what it covers
    (2, 60, 104, 2, False, 1),             # Lw = 1560 = 12*128 + 24   scale 0 of 480x832: 13 query tiles, ragged key tail
    (2, 60, 104, 2, True, 1),              # + cyclic shift, region mask in 3 of 4 windows
    (2, 120, 208, 8, True, 0),             # Lw = 390                  scale 1 of 480x832: 64 windows, 15 masked
    (2, 68, 120, 2, True, 1),              # Lw = 2040                 scale 0 of 544x960 (stereo self-attention)
    (2, 48, 64, 2, False, 1),              # Lw = 768                  384x512 (depth)
]


def _planes_from_rows(x, h, w, K, sh, sw):
    """[n, L, 128] fp32 -> window-major fp16 (hi, lo) planes [2, n, K*K, lp, 128] (what the projection epilogue writes)."""
    n = x.shape[0]
    lp = refops.planes_lp(h, w, K, K)
    rows = refops.window_rows(h, w, K, K, sh, sw, lp)
    hi = x.half()
    lo = (x - hi.float()).half()
    pl = torch.zeros((2, n, K * K * lp, C), dtype=torch.float16)
    pl[0][:, rows] = hi
    pl[1][:, rows] = lo
    return pl.view(2, n, K * K, lp, C)


@pytest.mark.parametrize("n,h,w,K,shift,kvs", FULL_ATTN_CASES)
def test_window_attention_fullsize_vs_oracle(n, h, w, K, shift, kvs):
    gen = g(5000 + h + K + int(shift))
    L = h * w
    q = torch.randn((n, L, C), generator=gen) * 1.5
    k = torch.randn((n, L, C), generator=gen) * 1.5
    v = torch.randn((n, L, C), generator=gen)
    wh, ww = h // K, w // K
    sh, sw = (wh // 2, ww // 2) if shift else (0, 0)
    mask = ops.MASK_SWIN if shift else ops.MASK_NONE
    ref = refops.window_attention(q, k, v, kvs, h, w, K, K, sh, sw, mask)
    # (a) fp32-rows entry point (split pass + kernel)
    got = OPS.window_attention(q.cuda(), k.cuda(), v.cuda(), kvs, h, w, K, K, sh, sw, mask)
    close(got, ref, 2e-5)
    # (b) operand-planes entry point, both output kinds
    assert ops.attention_planes_lp(h, w, K, K, sh, sw, mask) == refops.planes_lp(h, w, K, K)
    out_f = torch.zeros((n, L, C)).cuda()
    out_s = torch.zeros((2, n * L + 16, C), dtype=torch.float16).cuda()
    OPS.window_attention_planes(_planes_from_rows(q, h, w, K, sh, sw).cuda(), _planes_from_rows(k, h, w, K, sh, sw).cuda(),
                                _planes_from_rows(v, h, w, K, sh, sw).cuda(), n, kvs, h, w, K, K, sh, sw, mask, out_f, out_s)
    close(out_f, ref, 2e-5)
    close((out_s[0].float() + out_s[1].float())[:n * L].view(n, L, C), ref, 2e-5)
    assert out_s[:, n * L:].abs().max().item() == 0          # rows beyond the tokens are never written


@pytest.mark.parametrize("n,h,w,K,shift,c0,c1", [(2, 30, 52, 2, True, 0, 640), (1, 30, 52, 2, False, 0, 384),
                                                 (3, 32, 24, 1, False, 0, 128), (2, 60, 104, 2, True, 128, 384)])
def test_conv2d_tc_window_plane_output(n, h, w, K, shift, c0, c1):
    """The projection GEMM writing the attention's window-major operand planes (channels [c0, c1)) and fp32 rows for the
    rest; token rows padded to a multiple of 16 where n*h*w is not one."""
    gen = g(6000 + n + h + c1)
    L = h * w
    rows = n * L
    rp = (rows + 15) // 16 * 16
    cout = 640 if c1 > 128 else 128
    x = torch.randn((rows, C), generator=gen)
    wt = torch.randn((cout, C, 1, 1), generator=gen) * (2.0 / C) ** 0.5
    wp = ops.prep_conv_weight(wt, [C], cout)
    wh, ww = h // K, w // K
    sh, sw = (wh // 2, ww // 2) if shift else (0, 0)
    geom = (h, w, K, K, sh, sw, ops.MASK_SWIN if shift else ops.MASK_NONE)
    lp = refops.planes_lp(h, w, K, K)
    nops = (c1 - c0) // 128

    def run(dev, conv_fn, split_fn):
        src = torch.zeros((2, rp, C), dtype=torch.float16, device=dev)
        split_fn(x.to(dev), src, 0)
        y = torch.zeros((rp, cout), device=dev) if (c0 > 0 or c1 < cout) else None
        wd = torch.zeros((nops, 2, n, K * K, lp, C), dtype=torch.float16, device=dev)
        conv_fn(src, None, wp.to(dev), None, 1, 1, 0, 0, cout, 128, ops.CONV_LINEAR, ops.ACT_NONE, y, 0, None, 0, None, None,
                None, None, 1, rp, wd, geom, c0, c1, n)
        return (wd[:, 0].float() + wd[:, 1].float()).cpu(), None if y is None else y.cpu()

    ref_w, ref_y = run("cpu", refops.conv2d_tc, refops.split_planes)
    got_w, got_y = run("cuda", OPS.conv2d_tc, OPS.split_planes)
    close(got_w, ref_w, 2e-5)
    lw = wh * ww
    assert got_w[:, :, :, lw:].abs().max().item() == 0 if lp > lw else True      # window padding rows stay zero
    if ref_y is not None:
        close(got_y[:rows], ref_y[:rows], 2e-5)
        if c0 > 0:
            assert got_y[:, c0:c1].abs().max().item() == 0                       # those channels went to the planes only


def test_split_planes_into_padded_destination():
    x = torch.randn((37, C), generator=g(6100)) * 3
    dst = torch.zeros((2, 48, C), dtype=torch.float16).cuda()
    OPS.split_planes(x.cuda(), dst, 0)
    close((dst[0].float() + dst[1].float())[:37], x, 1e-6)
    assert dst[:, 37:].abs().max().item() == 0


def test_linear_over_row_range_of_larger_planes():
    """`rows` mode of conv2d_tc: the layer runs over the first rows of [2, R, cp] plane buffers (propagation projections on
    the first half of the streams), hi / lo planes R*cp apart; bias + fp32 and plane outputs."""
    gen = g(6200)
    R, rows = 96, 64
    x = torch.randn((R, C), generator=gen)
    wt = torch.randn((256, C, 1, 1), generator=gen) * 0.1
    bias = torch.randn(256, generator=gen) * 0.1
    wp = ops.prep_conv_weight(wt, [C], 256)

    def run(dev, conv_fn, split_fn):
        src = torch.zeros((2, R, C), dtype=torch.float16, device=dev)
        split_fn(x.to(dev), src, 0)
        y = torch.zeros((rows, 256), device=dev)
        ys = torch.zeros((2, rows + 16, 256), dtype=torch.float16, device=dev)
        conv_fn(src, None, wp.to(dev), bias.to(dev), 1, 1, 0, 0, 256, 128, ops.CONV_LINEAR, ops.ACT_NONE, y, 0, ys, 0, None, None,
                None, None, 1, rows)
        return y.cpu(), (ys[0].float() + ys[1].float()).cpu()

    ref_y, ref_s = run("cpu", refops.conv2d_tc, refops.split_planes)
    got_y, got_s = run("cuda", OPS.conv2d_tc, OPS.split_planes)
    close(got_y, ref_y, 2e-5)
    close(got_s, ref_s, 2e-5)
    close(got_y, torch.nn.functional.linear(x[:rows], wt.flatten(1), bias), 2e-5)


@pytest.mark.parametrize("mode", ["zr", "q"])
def test_conv2d_tc_preaccumulated_invariant_channels(mode):
    """SepConvGRU convolution with the loop-invariant input channels hoisted: conv(cat[a, b]) == conv_var(b) + pre, where
    pre = conv_fix(a) + bias is a fp32 tensor added to the accumulator before the gate math (um_conv_desc.pre)."""
    gen = g(7000 + len(mode))
    b, h, w = 2, 12, 40
    cout = 256 if mode == "zr" else 128
    wt = torch.randn((cout, 256, 1, 5), generator=gen) * (2.0 / (256 * 5)) ** 0.5
    bias = torch.randn(cout, generator=gen) * 0.1
    xa = torch.randn((b, h, w, 128), generator=gen)
    xb = torch.randn((b, h, w, 128), generator=gen)
    hh = torch.tanh(torch.randn((b, h, w, 128), generator=gen))
    zz = torch.sigmoid(torch.randn((b, h, w, 128), generator=gen))
    m = ops.CONV_GRU_ZR if mode == "zr" else ops.CONV_GRU_Q
    w_fix, w_var, w_all = (ops.prep_conv_weight(wt[:, :128], [128], cout), ops.prep_conv_weight(wt[:, 128:], [128], cout),
                           ops.prep_conv_weight(wt, [128, 128], cout))

    def run(dev, conv_fn, split_fn, hoisted):
        sa = torch.zeros((2, b, h, w, 128), dtype=torch.float16, device=dev)
        sb = torch.zeros((2, b, h, w, 128), dtype=torch.float16, device=dev)
        split_fn(xa.to(dev), sa, 0)
        split_fn(xb.to(dev), sb, 0)
        out_f = torch.zeros((b, h, w, 128), device=dev)
        out_s = torch.zeros((2, b, h, w, 128), dtype=torch.float16, device=dev)
        aux1 = zz.to(dev) if mode == "q" else None
        if hoisted:
            pre = torch.zeros((b, h, w, cout), device=dev)
            conv_fn(sa, None, w_fix.to(dev), bias.to(dev), 1, 5, 0, 2, cout, cout, ops.CONV_LINEAR, ops.ACT_NONE, pre, 0, None, 0, None, None)
            conv_fn(sb, None, w_var.to(dev), None, 1, 5, 0, 2, cout, cout, m, 0, out_f, 0, out_s, 0, hh.to(dev), aux1, None, None, 1, 0,
                    None, None, 0, 0, 0, pre)
        else:
            conv_fn(sa, sb, w_all.to(dev), bias.to(dev), 1, 5, 0, 2, cout, cout, m, 0, out_f, 0, out_s, 0, hh.to(dev), aux1)
        return out_f.cpu(), (out_s[0].float() + out_s[1].float()).cpu()

    ref_f, ref_s = run("cpu", refops.conv2d_tc, refops.split_planes, True)
    got_f, got_s = run("cuda", OPS.conv2d_tc, OPS.split_planes, True)
    whole_f, whole_s = run("cuda", OPS.conv2d_tc, OPS.split_planes, False)
    close(got_f, ref_f, 2e-5)
    close(got_s, ref_s, 2e-5)
    close(got_f, whole_f, 2e-5)          # hoisting changes the summation order only
    close(got_s, whole_s, 2e-5)
