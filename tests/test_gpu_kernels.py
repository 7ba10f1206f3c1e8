"""Kernel-level parity (needs a B200): every C-ABI op against a plain PyTorch fp32 statement of the same op on
identical (bf16-rounded) inputs.  Integer paths are bit-exact; floating point within the stated tolerance."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL_ACT = 1e-2      # BASELINE.md section 5: forward activations <= 1e-2 relative error (bf16 in / fp32 accumulate)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def bf(x):
    return x.to(torch.bfloat16).float()


@pytest.fixture(scope="module")
def S():
    from seg2eye_b200 import _lib as L, ops
    L.lib()
    return L, ops


def nhwc(x):  # NCHW fp32 cpu -> NHWC bf16 cuda
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()


def nchw(y):  # NHWC cuda -> NCHW fp32 cpu
    return y.float().permute(0, 3, 1, 2).cpu()


# ------------------------------------------------------------------------------------------ integer path
def test_onehot_and_nearest_bit_exact(S):
    L, ops = S
    ints = dict(np.load(os.path.join(GOLD, "ref_ints.npz")))
    for key_l, key_o in (("label", "onehot"), ("rand_label", "rand_onehot")):
        lab = torch.from_numpy(ints[key_l]).cuda()
        oh = ops.one_hot(lab, 4)
        assert np.array_equal(oh.cpu().numpy().astype(np.uint8), ints[key_o])
    seg = torch.from_numpy(ints["onehot"]).float().cuda()
    for k, v in ints.items():
        if k.startswith("nearest_"):
            h, w = [int(s) for s in k.split("_")[1].split("x")]
            out = ops.seg_nearest(seg, h, w)
            assert np.array_equal(nchw(out).numpy().astype(np.uint8), v), k
    seg2 = torch.from_numpy(ints["rand_onehot"]).float().cuda()
    out = ops.seg_nearest(seg2, 9, 13)
    assert np.array_equal(nchw(out).numpy().astype(np.uint8), ints["rand_nearest_9x13"])


def test_layout_roundtrip(S):
    L, ops = S
    x = torch.randn(2, 5, 7, 9)
    y = ops.ToNHWCFn.apply(x.cuda())
    assert torch.equal(y.cpu().float(), bf(x).permute(0, 2, 3, 1))
    z = ops.ToNCHWFn.apply(y)
    assert torch.equal(z.cpu(), bf(x))


# ------------------------------------------------------------------------------------------ convolutions
def conv_case(S, impl, B, Cin, Cout, H, W, k, stride, pad, act=0, sn=False, n_w=1, seed=0, bias=True):
    L, ops = S
    g = torch.Generator().manual_seed(seed)
    x = bf(torch.randn(B, Cin, H, W, generator=g))
    ws = [bf(torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5) for _ in range(n_w)]
    bs = [torch.randn(Cout, generator=g) * 0.1 for _ in range(n_w)] if bias else []
    inv_sigma = 0.7 if sn else 1.0
    # reference (CPU fp32)
    xr = x.clone().requires_grad_()
    wr = [w.clone().requires_grad_() for w in ws]
    br = [b.clone().requires_grad_() for b in bs]
    yr = F.conv2d(xr, torch.cat(wr, 0) * inv_sigma, torch.cat(br, 0) if bias else None, stride=stride, padding=pad)
    if act == 1:
        yr = F.leaky_relu(yr, 0.2)
    elif act == 2:
        yr = F.relu(yr)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    # ours
    xc = nhwc(x).requires_grad_()
    wc = [w.cuda().requires_grad_() for w in ws]
    bc = [b.cuda().requires_grad_() for b in bs]
    cfg = ops.ConvCfg(k, k, stride, pad, act)
    snt = None
    if sn:
        # u, v only enter the backward; choose them so that the sigma chain-rule term is exercised
        u = F.normalize(torch.randn(Cout, generator=g), dim=0).cuda()
        v = F.normalize(torch.randn(Cin * k * k, generator=g), dim=0).cuda()
        snt = (u, v, torch.tensor([inv_sigma], device="cuda"))
    with ops.force_impl(impl):
        y = ops.tap_conv(xc, cfg, tuple(wc), tuple(bc), snt)
        y.backward(nhwc(dy))
    torch.cuda.synchronize()
    assert rel(nchw(y), yr) < TOL_ACT, ("fwd", rel(nchw(y), yr))
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT, ("dgrad", rel(nchw(xc.grad), xr.grad))
    for i in range(n_w):
        gw_ref = wr[i].grad
        if sn:
            # y = conv(x, W_orig) * inv_sigma with sigma = u^T W v  =>  dW_orig = is*(G - is*<G,W> u v^T), G = dL/dW_eff
            G = wr[i].grad / inv_sigma
            uv = torch.outer(u.cpu(), v.cpu()).view_as(G)
            gw_ref = inv_sigma * (G - inv_sigma * (G * ws[i]).sum() * uv)
        assert rel(wc[i].grad, gw_ref) < TOL_ACT, ("wgrad", i, rel(wc[i].grad, gw_ref))
        if bias:
            assert rel(bc[i].grad, br[i].grad) < TOL_ACT, ("bgrad", i, rel(bc[i].grad, br[i].grad))


SIMT_CASES = [
    # B, Cin, Cout, H, W, k, stride, pad, act
    (2, 4, 128, 10, 8, 3, 1, 1, 2),      # mlp_shared-like (+ReLU)
    (2, 4, 32, 10, 8, 3, 1, 1, 0),       # G.fc-like
    (1, 16, 1, 20, 16, 3, 1, 1, 0),      # conv_img-like (Cout = 1)
    (2, 5, 16, 21, 17, 4, 2, 2, 1),      # D model0 (4x4 s2 p2 + LeakyReLU), odd size
    (2, 32, 1, 11, 9, 4, 1, 2, 0),       # D model4 (Cout = 1, 4x4 s1 p2)
    (2, 1, 16, 32, 32, 3, 2, 1, 0),      # E layer0 (3x3 s2 p1, Cin = 1)
    (1, 24, 40, 9, 7, 1, 1, 0, 0),       # 1x1 with ragged channel counts
    (2, 16, 32, 13, 11, 4, 2, 2, 0),     # 4x4 s2 p2 mid layer, odd size
    (2, 64, 1, 21, 18, 3, 1, 1, 0),      # conv_img at ngf=64 (mma.sync tile kernel; data / weight gradient on mma.sync too)
    (1, 64, 1, 19, 141, 3, 1, 1, 0),     # the same, several tiles per row, ragged
    (2, 128, 1, 19, 21, 4, 1, 2, 0),     # PatchGAN head shape on the generic thin-output kernels
]


@pytest.mark.parametrize("case", SIMT_CASES)
def test_conv_simt_vs_torch(S, case):
    L, ops = S
    conv_case(S, L.IMPL_SIMT, *case)


TC_CASES = [
    (2, 128, 128, 10, 8, 3, 1, 1, 0),      # gamma|beta-like, tiny map (tile spans batch)
    (1, 64, 64, 20, 16, 3, 1, 1, 0),
    (2, 128, 256, 20, 16, 3, 1, 1, 0),     # BN = 256
    (1, 256, 128, 40, 32, 3, 1, 1, 0),
    (1, 128, 64, 40, 32, 1, 1, 0, 0),      # 1x1 shortcut
    (3, 64, 128, 21, 17, 4, 2, 2, 0),      # D 4x4 s2 p2 (space-to-depth, Cin' = 256), odd size
    (2, 64, 128, 11, 9, 4, 1, 2, 0),       # D 4x4 s1 p2: output larger than input
    (2, 64, 128, 32, 32, 3, 2, 1, 0),      # E 3x3 s2 p1
    (1, 64, 72, 16, 8, 3, 1, 1, 1),        # Cout not a multiple of 64, fused LeakyReLU
    (2, 128, 512, 16, 16, 3, 1, 1, 0),     # wgrad orientation swapped (Cout > Cin): accumulator [Cin x Cout], N = 256
    (2, 128, 64, 24, 16, 3, 1, 1, 0),      # wgrad swapped because Cout < 128 <= Cin
    (2, 64, 64, 24, 16, 3, 1, 1, 0),
]


@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tcgen05_vs_torch(S, case):
    L, ops = S
    conv_case(S, L.IMPL_TC, *case)


MT_WGRAD_CASES = [
    (2, 64, 64, 24, 16, 3, 1, 1, 0),       # M = 128 half empty, N = 64
    (2, 128, 64, 24, 16, 3, 1, 1, 0),      # swapped orientation
    (2, 64, 128, 24, 16, 3, 1, 1, 0),      # swapped (Cout > Cin)
    (2, 128, 128, 24, 16, 3, 1, 1, 0),     # N = 128: three 128-column accumulators
    (1, 64, 64, 37, 29, 3, 1, 1, 0),       # ragged map: partial pixel tiles at the right / bottom edge
    (3, 128, 128, 40, 48, 3, 1, 1, 0),     # many pixel tiles per CTA, several split-K slices
    (2, 64, 128, 11, 9, 4, 1, 2, 0),       # 16 taps: last group has one tap
]


@pytest.mark.parametrize("case", MT_WGRAD_CASES)
def test_conv_tcgen05_multitap_wgrad(S, case):
    """Weight gradients of narrow layers (N side < 256): tapconv_wgrad_mt_kernel (several taps per CTA against one staged dY
    tile, the default) and, with debug key 5 = 1, the one-tap-per-CTA kernel it replaced."""
    L, ops = S
    conv_case(S, L.IMPL_TC, *case)
    L.call("s2e_debug_set", 5, 1)
    try:
        conv_case(S, L.IMPL_TC, *case)
    finally:
        L.call("s2e_debug_set", 5, 0)


def test_conv_tcgen05_fused_gamma_beta_and_spectral(S):
    L, ops = S
    conv_case(S, L.IMPL_TC, 2, 128, 64, 20, 16, 3, 1, 1, 0, n_w=2)           # two weights packed along Cout
    conv_case(S, L.IMPL_TC, 2, 64, 128, 20, 16, 3, 1, 1, 0, sn=True)         # 1/sigma epilogue + chain rule
    conv_case(S, L.IMPL_SIMT, 2, 16, 24, 12, 10, 4, 2, 2, 0, sn=True, bias=False)


@pytest.mark.parametrize("impl_name", ["tc", "simt"])
def test_seg_im2col_conv_matches_conv3x3(S, impl_name):
    """SPADE's mlp_shared on the 64-channel im2col of the (nearest-resized) segmap == ReLU(conv3x3(seg))."""
    L, ops = S
    g = torch.Generator().manual_seed(9)
    B, C, Hs, Ws, hd, wd, Cout = 2, 4, 40, 32, 20, 16, 128
    seg = F.one_hot(torch.randint(0, C, (B, Hs, Ws), generator=g), C).permute(0, 3, 1, 2).float()
    w = bf(torch.randn(Cout, C, 3, 3, generator=g) / 6.0)
    b = torch.randn(Cout, generator=g) * 0.1
    segr = F.interpolate(seg, size=(hd, wd), mode="nearest")
    wr, br = w.clone().requires_grad_(), b.clone().requires_grad_()
    yr = F.relu(F.conv2d(segr, wr, br, padding=1))
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    col = ops.seg_im2col(seg.cuda(), hd, wd)
    # bit-exact im2col: channel (r*3+s)*C + c
    ref_col = F.unfold(segr, 3, padding=1).view(B, C, 9, hd, wd).permute(0, 3, 4, 2, 1).reshape(B, hd, wd, 9 * C)
    assert torch.equal(col[..., :9 * C].float().cpu(), ref_col) and float(col[..., 9 * C:62].abs().max()) == 0.0
    assert bool((col[..., 62:] == 1).all())    # constant-one channels: carry the bias (and its gradient) through the GEMM
    wc, bc = w.cuda().requires_grad_(), b.cuda().requires_grad_()
    with ops.force_impl(L.IMPL_TC if impl_name == "tc" else L.IMPL_SIMT):
        y = ops.SegConvFn.apply(col, wc, bc, L.ACT_RELU)
        y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < TOL_ACT
    assert rel(wc.grad, wr.grad) < TOL_ACT and rel(bc.grad, br.grad) < TOL_ACT


@pytest.mark.parametrize("impl_name", ["tc", "simt"])
def test_relu_backward_fused_into_dgrad_epilogue(S, impl_name):
    """conv(relu(a)) with relu_in=True: the gradient returned for relu(a) is already masked by (relu(a) > 0)."""
    L, ops = S
    g = torch.Generator().manual_seed(11)
    B, Cin, Cout, H, W = 2, 128, 64, 12, 20
    a = bf(torch.randn(B, Cin, H, W, generator=g))
    w = bf(torch.randn(Cout, Cin, 3, 3, generator=g) / (Cin * 9) ** 0.5)
    ar, wr = a.clone().requires_grad_(), w.clone().requires_grad_()
    yr = F.conv2d(F.relu(ar), wr, None, padding=1)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = nhwc(F.relu(a)).requires_grad_()
    wc = w.cuda().requires_grad_()
    with ops.force_impl(L.IMPL_TC if impl_name == "tc" else L.IMPL_SIMT):
        y = ops.tap_conv(xc, ops.ConvCfg(3, 3, 1, 1, 0, True), (wc,), ())
        y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < TOL_ACT
    assert rel(nchw(xc.grad), ar.grad) < TOL_ACT          # masked gradient == gradient w.r.t. the pre-ReLU tensor
    assert float((nchw(xc.grad)[F.relu(a) <= 0]).abs().max()) == 0.0
    assert rel(wc.grad, wr.grad) < TOL_ACT


def test_channel_padded_input_runs_d_first_layer_on_tensor_cores(S):
    """D model0 (5 -> 64, 4x4 s2 p2, LeakyReLU): activations zero-padded to 16 channels, weights keep their 5."""
    L, ops = S
    g = torch.Generator().manual_seed(13)
    B, Cin, Cpad, Cout, H, W = 2, 5, 16, 64, 21, 18
    x = bf(torch.randn(B, Cin, H, W, generator=g))
    w = bf(torch.randn(Cout, Cin, 4, 4, generator=g) / (Cin * 16) ** 0.5)
    b = torch.randn(Cout, generator=g) * 0.1
    xr, wr, br = x.clone().requires_grad_(), w.clone().requires_grad_(), b.clone().requires_grad_()
    yr = F.leaky_relu(F.conv2d(xr, wr, br, stride=2, padding=2), 0.2)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xp = torch.zeros(B, Cpad, H, W)
    xp[:, :Cin] = x
    xc = nhwc(xp).requires_grad_()
    wc, bc = w.cuda().requires_grad_(), b.cuda().requires_grad_()
    y = ops.tap_conv(xc, ops.ConvCfg(4, 4, 2, 2, L.ACT_LRELU, False, Cpad), (wc,), (bc,))
    y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < TOL_ACT
    assert rel(nchw(xc.grad)[:, :Cin], xr.grad) < TOL_ACT and float(nchw(xc.grad)[:, Cin:].abs().max()) == 0.0
    assert rel(wc.grad, wr.grad) < TOL_ACT and rel(bc.grad, br.grad) < TOL_ACT


def test_conv_tcgen05_large_k_many_tiles(S):
    L, ops = S
    conv_case(S, L.IMPL_TC, 4, 512, 512, 20, 16, 3, 1, 1, 0, seed=3)         # K = 4608, two N tiles, 20 work items: one per CTA


# ------------------------------------------------------------------------------------------ spectral norm
def test_spectral_power_iteration(S):
    L, ops = S
    g = torch.Generator().manual_seed(1)
    w = torch.randn(48, 20, 3, 3, generator=g)
    u = F.normalize(torch.randn(48, generator=g), dim=0)
    v = F.normalize(torch.randn(180, generator=g), dim=0)
    wm = w.view(48, -1)
    v1 = F.normalize(torch.mv(wm.t(), u), dim=0, eps=1e-12)
    u1 = F.normalize(torch.mv(wm, v1), dim=0, eps=1e-12)
    sigma = torch.dot(u1, torch.mv(wm, v1))
    uc, vc = u.cuda(), v.cuda()
    inv = ops.spectral_inv_sigma(w.cuda(), uc, vc, True)
    assert rel(uc, u1) < 1e-5 and rel(vc, v1) < 1e-5 and abs(float(inv) * float(sigma) - 1) < 1e-5
    # eval mode: buffers untouched
    u2, v2 = u.cuda(), v.cuda()
    inv2 = ops.spectral_inv_sigma(w.cuda(), u2, v2, False)
    assert torch.equal(u2.cpu(), u) and torch.equal(v2.cpu(), v)
    assert abs(float(inv2) * float(torch.dot(u, torch.mv(wm, v))) - 1) < 1e-5


# ------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("per_sample,act,C", [(False, 1, 64), (False, 0, 1024), (True, 1, 48), (False, 1, 8)])
def test_spade_style_fwd_bwd(S, per_sample, act, C):
    L, ops = S
    g = torch.Generator().manual_seed(2)
    B, H, W = 3, 12, 10
    x = bf(torch.randn(B, C, H, W, generator=g) * 1.5 + 0.3)
    gam = bf(torch.randn(B, C, H, W, generator=g) * 0.5)
    bet = bf(torch.randn(B, C, H, W, generator=g) * 0.5)
    style = torch.randn(B, 2 * C, generator=g) * 0.5
    rm0, rv0 = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    xr, gr, br, sr = [t.clone().requires_grad_() for t in (x, gam, bet, style)]
    if per_sample:
        xn = F.instance_norm(xr, eps=1e-5)
        rm, rv = rm0.clone(), rv0.clone()
    else:
        rm, rv = rm0.clone(), rv0.clone()
        xn = F.batch_norm(xr, rm, rv, training=True, momentum=0.1, eps=1e-5)
    out_r = 0.5 * (xn * (1 + gr) + br + xr * (1 + sr[:, :C, None, None]) + sr[:, C:, None, None])
    if act:
        out_r = F.leaky_relu(out_r, 0.2)
    dout = bf(torch.randn(out_r.shape, generator=g))
    out_r.backward(dout)

    xc = nhwc(x).requires_grad_()
    gbc = torch.cat([nhwc(gam), nhwc(bet)], dim=3).contiguous().requires_grad_()
    sc = style.cuda().requires_grad_()
    rmc, rvc, nbt = rm0.cuda(), rv0.cuda(), torch.tensor(3, device="cuda")
    cfg = ops.NormCfg(per_sample, act, True, 0.1, 1e-5)
    seen = {}
    xin, gbin = ops.AddFn.apply(xc, torch.zeros_like(xc)), ops.AddFn.apply(gbc, torch.zeros_like(gbc))   # non-leaf inputs
    xin.register_hook(lambda t: seen.__setitem__("x", t))
    gbin.register_hook(lambda t: seen.__setitem__("gb", t))
    if per_sample:
        out = ops.SpadeStyleFn.apply(xin, gbin, sc, cfg, None, None, None)
    else:
        out = ops.SpadeStyleFn.apply(xin, gbin, sc, cfg, rmc, rvc, nbt)
    out.backward(nhwc(dout))
    torch.cuda.synchronize()
    assert rel(nchw(out), out_r) < 5e-3
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT
    assert rel(nchw(gbc.grad[..., :C]), gr.grad) < TOL_ACT
    assert rel(nchw(gbc.grad[..., C:]), br.grad) < TOL_ACT
    assert rel(sc.grad, sr.grad) < TOL_ACT
    if not per_sample:
        assert rel(rmc, rm) < 1e-4 and rel(rvc, rv) < 1e-4 and int(nbt) == 4
    # per-channel sums of dgamma | dbeta and of dx that ride on the gradients (bias gradients of the neighbouring convs)
    s_gb, s_x = seen["gb"]._s2e_chsum, seen["x"]._s2e_chsum
    ref_gb = torch.cat([gr.grad.sum(dim=(0, 2, 3)), br.grad.sum(dim=(0, 2, 3))])
    assert rel(s_gb, ref_gb) < 2e-3
    ref_x = xr.grad.sum(dim=(0, 2, 3))
    assert float((s_x.cpu() - ref_x).abs().max()) < 2e-3 * float(xr.grad.abs().sum(dim=(0, 2, 3)).max())


@pytest.mark.parametrize("act,C", [(1, 64), (0, 512), (1, 16)])
def test_instance_norm_fwd_bwd(S, act, C):
    L, ops = S
    g = torch.Generator().manual_seed(4)
    x = bf(torch.randn(3, C, 9, 11, generator=g) * 2 + 1)
    xr = x.clone().requires_grad_()
    yr = F.instance_norm(xr, eps=1e-5)
    if act:
        yr = F.leaky_relu(yr, 0.2)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = nhwc(x).requires_grad_()
    y = ops.InstNormFn.apply(xc, act)
    y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < 5e-3
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT


@pytest.mark.parametrize("per_sample", [False, True])
def test_statistics_of_large_mean_channels(S, per_sample):
    """Per-channel mean / 1/sqrt(var + eps) of channels whose mean is 200 standard deviations away from zero: the shifted
    accumulation (pivot = first pixel) keeps ~1e-6 where raw E[x^2] - E[x]^2 moments from fp32 partial sums lose (mean/sigma)^2
    of their precision.  Also the plain channel sums derived from the shifted ones (bias gradients)."""
    L, ops = S
    g = torch.Generator().manual_seed(8)
    B, H, W, C = 3, 96, 80, 64
    x = (torch.randn(B, H, W, C, generator=g) * 0.25 + 50.0 * (1 + torch.arange(C).float() / C)).to(torch.bfloat16).cuda()
    cfg = ops.NormCfg(per_sample, L.ACT_NONE, True, 0.1, 1e-5)
    mean, rstd, _ = ops.spade_statistics(x, cfg, None, None, None, False)
    xd = x.double()
    dims = (1, 2) if per_sample else (0, 1, 2)
    m_ref = xd.mean(dim=dims)
    v_ref = xd.var(dim=dims, unbiased=False)
    r_ref = 1.0 / torch.sqrt(v_ref + 1e-5)
    assert float(((mean.double().view_as(m_ref) - m_ref).abs() / m_ref.abs()).max()) < 1e-6
    assert float(((rstd.double().view_as(r_ref) - r_ref).abs() / r_ref).max()) < 1e-4
    sums = ops.channel_sums(x.view(-1, C), B, H * W, C)
    s_ref = xd.sum(dim=(0, 1, 2))
    assert float(((sums.double() - s_ref).abs() / s_ref.abs()).max()) < 1e-6


@pytest.mark.parametrize("act,C,H,W", [(1, 128, 161, 97), (1, 512, 42, 26), (2, 256, 33, 40), (0, 2048, 8, 8), (1, 4096, 4, 4)])
def test_instance_norm_streaming_paths(S, act, C, H, W):
    """The discriminator's / encoder's shapes (discriminator.py:34-37, encoder.py:23-38): several pixels in flight per thread,
    more channel groups than threads, activation sign recomputed from x in the backward pass (large-mean channels included)."""
    L, ops = S
    g = torch.Generator().manual_seed(6)
    x = bf(torch.randn(2, C, H, W, generator=g) * torch.rand(1, C, 1, 1, generator=g) * 3 + torch.randn(1, C, 1, 1, generator=g) * 4)
    xr = x.clone().requires_grad_()
    yr = F.instance_norm(xr, eps=1e-5)
    yr = F.leaky_relu(yr, 0.2) if act == 1 else (F.relu(yr) if act == 2 else yr)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = nhwc(x).requires_grad_()
    y = ops.InstNormFn.apply(xc, act)
    y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < 5e-3
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT, rel(nchw(xc.grad), xr.grad)


@pytest.mark.parametrize("B,C,H,W", [(6, 128, 21, 17), (4, 512, 9, 11), (32, 256, 40, 24), (2, 4096, 3, 3)])
def test_feature_matching_sum_fused_into_instance_norm(S, B, C, H, W):
    """Inside ops.fm_pair_sums() an InstanceNorm layer fed with a [fake ; real] batch normalises both halves in one block and
    reduces sum |y_fake - y_real| on the way (pix2pix_model.py:233-241): same output bits as the plain kernel, same loss value
    and gradient as the separate reduction (ops.HalvesLossFn)."""
    L, ops = S
    from seg2eye_b200.models.networks.layers import InstanceNorm2d
    g = torch.Generator().manual_seed(23)
    x0 = (torch.randn(B, H, W, C, generator=g) * 2 + 0.5).to(torch.bfloat16).cuda()
    norm = InstanceNorm2d(C, L.ACT_LRELU)
    dy = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16).cuda()
    out = {}
    for fused in (False, True):
        x = x0.clone().requires_grad_()
        if fused:
            with ops.fm_pair_sums():
                y = norm.forward_nhwc(x)
            assert hasattr(y, "_s2e_fm_sum")
            term = ops.HalvesPresummedFn.apply(y, y._s2e_fm_sum[0], L.RED_L1, 2.0 / y.numel())
        else:
            y = norm.forward_nhwc(x)
            assert not hasattr(y, "_s2e_fm_sum")
            term = ops.HalvesLossFn.apply(y, L.RED_L1, 2.0 / y.numel())
        (term.sum() * 3.0 + (y.float() * dy.float()).sum() * 1e-3).backward()
        out[fused] = (y.detach().clone(), float(term.detach()), x.grad.float().clone())
    assert torch.equal(out[True][0], out[False][0])
    ref = float((out[False][0][:B // 2].float() - out[False][0][B // 2:].float()).abs().mean())
    assert abs(out[True][1] - ref) < 1e-4 * ref and abs(out[False][1] - ref) < 1e-4 * ref, (out[True][1], out[False][1], ref)
    assert rel(out[True][2].cpu(), out[False][2].cpu()) < 1e-5


# ------------------------------------------------------------------------------------------ resampling / elementwise
def test_upsample_avgpool_bilinear_add_act(S):
    L, ops = S
    g = torch.Generator().manual_seed(5)
    x = bf(torch.randn(2, 16, 5, 7, generator=g))
    xr = x.clone().requires_grad_()
    yr = F.interpolate(xr, scale_factor=2, mode="nearest")
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = nhwc(x).requires_grad_()
    y = ops.Upsample2xFn.apply(xc)
    y.backward(nhwc(dy))
    assert torch.equal(nchw(y), yr.detach())
    assert rel(nchw(xc.grad), xr.grad) < 5e-3

    for (H, W, Cp) in [(12, 10, 5), (13, 9, 5), (13, 10, 16)]:
        x = bf(torch.randn(2, Cp, H, W, generator=g))
        xr = x.clone().requires_grad_()
        yr = F.avg_pool2d(xr, kernel_size=3, stride=2, padding=[1, 1], count_include_pad=False)
        dy = bf(torch.randn(yr.shape, generator=g))
        yr.backward(dy)
        xc = nhwc(x).requires_grad_()
        y = ops.AvgPool3s2Fn.apply(xc)
        y.backward(nhwc(dy))
        assert rel(nchw(y), yr) < 5e-3 and rel(nchw(xc.grad), xr.grad) < 5e-3

    x = torch.rand(3, 1, 40, 32, generator=g) * 2 - 1
    xr = x.clone().requires_grad_()
    yr = F.interpolate(xr, size=(64, 64), mode="bilinear", align_corners=False)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = x.cuda().requires_grad_()
    y = ops.BilinearFn.apply(xc, (64, 64))
    y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < 5e-3 and rel(xc.grad, xr.grad) < 5e-3

    a, b = bf(torch.randn(2, 8, 3, 5, generator=g)), bf(torch.randn(2, 8, 3, 5, generator=g))
    assert rel(nchw(ops.AddFn.apply(nhwc(a), nhwc(b))), a + b) < 5e-3
    ac = nhwc(a).requires_grad_()
    z = ops.ActFn.apply(ac, L.ACT_LRELU)
    z.backward(nhwc(b))
    ar = a.clone().requires_grad_()
    F.leaky_relu(ar, 0.2).backward(b)
    assert rel(nchw(z), F.leaky_relu(a, 0.2)) < 5e-3 and rel(nchw(ac.grad), ar.grad) < 5e-3


def test_d_input_tanh_linear_losses_adam(S):
    L, ops = S
    g = torch.Generator().manual_seed(6)
    B, H, W = 2, 6, 5
    seg = F.one_hot(torch.randint(0, 4, (B, H, W), generator=g), 4).permute(0, 3, 1, 2).float()
    fake, real = torch.rand(B, 1, H, W, generator=g) * 2 - 1, torch.rand(B, 1, H, W, generator=g) * 2 - 1
    fc = fake.cuda().requires_grad_()
    out = ops.MakeDInputFn.apply(seg.cuda(), fc, real.cuda())
    ref = torch.cat([torch.cat([seg, fake], 1), torch.cat([seg, real], 1)], 0)
    assert rel(nchw(out), bf(ref)) < 1e-6
    dout = bf(torch.randn(out.shape, generator=g))
    out.backward(dout.cuda().to(torch.bfloat16))
    assert rel(fc.grad, dout[:B, :, :, 4].unsqueeze(1)) < 1e-6

    x = bf(torch.randn(B, 1, H, W, generator=g))
    xc = nhwc(x).requires_grad_()
    y = ops.TanhFn.apply(xc)
    dy = torch.randn(B, 1, H, W, generator=g)
    y.backward(dy.cuda())
    xr = x.clone().requires_grad_()
    torch.tanh(xr).backward(dy)
    assert rel(y, torch.tanh(x)) < 1e-5 and rel(nchw(xc.grad), xr.grad) < 5e-3

    # FC 16 -> 2C with LeakyReLU (normalization.py:134-141)
    w, b, xin = torch.randn(24, 16, generator=g) * 0.25, torch.randn(24, generator=g) * 0.1, torch.randn(3, 16, generator=g)
    wr, br_, xr = [t.clone().requires_grad_() for t in (w, b, xin)]
    yr = F.leaky_relu(F.linear(xr, wr, br_), 0.2)
    dy = torch.randn(3, 24, generator=g)
    yr.backward(dy)
    wc, bc, xc = [t.cuda().requires_grad_() for t in (w, b, xin)]
    y = ops.LinearFn.apply(xc, wc, bc, L.ACT_LRELU, 0)
    y.backward(dy.cuda())
    for a_, b_ in ((y, yr), (wc.grad, wr.grad), (bc.grad, br_.grad), (xc.grad, xr.grad)):
        assert rel(a_, b_) < 1e-5
    # encoder head: LeakyReLU + NCHW flatten of an NHWC feature (encoder.py:64-68)
    feat = bf(torch.randn(3, 8, 4, 4, generator=g))
    w2, b2 = torch.randn(16, 128, generator=g) * 0.1, torch.randn(16, generator=g) * 0.1
    fr, w2r, b2r = [t.clone().requires_grad_() for t in (feat, w2, b2)]
    yr = F.linear(F.leaky_relu(fr, 0.2).view(3, -1), w2r, b2r)
    dy = torch.randn(3, 16, generator=g)
    yr.backward(dy)
    fcu = nhwc(feat).requires_grad_()
    w2c, b2c = w2.cuda().requires_grad_(), b2.cuda().requires_grad_()
    y = ops.LinearFn.apply(fcu, w2c, b2c, L.ACT_NONE, 16)
    y.backward(dy.cuda())
    assert rel(y, yr) < 1e-5 and rel(w2c.grad, w2r.grad) < 1e-5 and rel(b2c.grad, b2r.grad) < 1e-5
    assert rel(nchw(fcu.grad), fr.grad) < 5e-3

    # loss reductions
    p = bf(torch.randn(2, 1, 9, 7, generator=g))
    p = bf(torch.where((p.abs() - 1).abs() < 1e-2, p * 1.1, p))   # keep away from the hinge kink (sub-gradient ties)
    q = bf(torch.randn(2, 1, 9, 7, generator=g))
    for kind, fn in ((L.RED_SUM, lambda t: t.sum()), (L.RED_HINGE_REAL, lambda t: torch.clamp(t - 1, max=0).sum()),
                     (L.RED_HINGE_FAKE, lambda t: torch.clamp(-t - 1, max=0).sum()),
                     (L.RED_L1, lambda t: (t - q).abs().sum()), (L.RED_L2, lambda t: ((t - q) ** 2).sum())):
        for dt in (torch.float32, torch.bfloat16):
            pr = p.clone().requires_grad_()
            lr_ = fn(pr) * 0.37
            lr_.backward()
            pc = p.cuda().to(dt).requires_grad_()
            yq = q.cuda().to(dt) if kind in (L.RED_L1, L.RED_L2) else None
            lo = ops.reduce_loss(pc, yq, kind, 0.37)
            lo.sum().backward()
            assert abs(float(lo) - float(lr_)) < 1e-4 * max(1.0, abs(float(lr_))), (kind, dt)
            assert rel(pc.grad.float(), pr.grad) < 5e-3, (kind, dt)

    # Adam (torch.optim.Adam semantics, betas (0, 0.9) as under TTUR)
    from seg2eye_b200 import optim
    p0, gr = torch.randn(1000, generator=g), torch.randn(3, 1000, generator=g)
    pr = p0.clone().requires_grad_()
    pc = p0.cuda().requires_grad_()
    o_r = torch.optim.Adam([pr], lr=1e-3, betas=(0.0, 0.9))
    o_c = optim.Adam([pc], lr=1e-3, betas=(0, 0.9))
    for i in range(3):
        pr.grad = gr[i].clone()
        pc.grad = gr[i].cuda()
        o_r.step()
        o_c.step()
    assert rel(pc, pr) < 1e-6


def test_space_to_depth_roundtrip(S):
    L, ops = S
    x = bf(torch.randn(2, 3, 7, 9))
    xc = nhwc(x)
    y = ops.space_to_depth(xc)
    assert y.shape == (2, 4, 5, 12)
    xp = F.pad(x, (0, 1, 0, 1))
    ref = torch.stack([xp[:, :, i::2, j::2] for i in (0, 1) for j in (0, 1)], dim=1).reshape(2, 12, 4, 5)
    assert torch.equal(nchw(y), ref)


# ------------------------------------------------------------------------------------------ multi-tensor ops
def test_pack_weight_multi_equals_single_calls(S):
    """One multi-tensor launch == the per-tensor s2e_pack_weight / s2e_pack_weight_im2col3x3 calls, bit for bit, for
    every geometry on the path (3x3, 1x1, 4x4 s2 p2 with channel padding, 3x3 s2 p1, 4x4 s1 p2, gamma|beta pairs)."""
    L, ops = S
    g = torch.Generator().manual_seed(5)
    cases = [(3, 3, 1, 1, 0, (72, 40), 24), (1, 1, 1, 0, 0, (64,), 136), (4, 4, 2, 2, 16, (64,), 5), (3, 3, 2, 1, 0, (32,), 8),
             (4, 4, 1, 2, 0, (8,), 64)]
    ops._pack_cache.clear()
    expect = []
    for kh, kw, st, pad, cpad, couts, cin in cases:
        ws = [torch.randn(co, cin, kh, kw, generator=g).cuda() for co in couts]
        cfg = ops.ConvCfg(kh, kw, st, pad, L.ACT_NONE, False, cpad)
        for tr in (False, True):
            cin_eff = max(cin, cpad) * (4 if st == 2 else 1)
            n = len(ops.conv_taps(cfg)) * sum(couts) * cin_eff
            ref = torch.zeros(n, dtype=torch.bfloat16, device="cuda")
            off = 0
            for w in ws:
                L.call("s2e_pack_weight", L.ptr(w), w.shape[0], cin, kh, kw, st, pad, int(tr), sum(couts), off, cpad, L.ptr(ref),
                       L.stream())
                off += w.shape[0]
            got = ops.packed_weights(tuple(ws), cfg, tr)
            assert torch.equal(got, ref), (kh, st, tr)
            expect.append((ws, cfg, tr))
    wseg = torch.randn(128, 4, 3, 3, generator=g).cuda()
    ref = torch.empty(128 * 64, dtype=torch.bfloat16, device="cuda")
    L.call("s2e_pack_weight_im2col3x3", L.ptr(wseg), 128, 4, L.ptr(ref), L.stream())
    assert torch.equal(ops.packed_weight_im2col(wseg), ref)
    # change every master weight behind torch's back (as the Adam kernel does) and re-pack everything in one call
    n0 = L.launches
    for ws, _, _ in expect:
        for w in ws:
            w.detach().view(-1)[::3] += 1.0
    ops.mark_updated([w for ws, _, _ in expect for w in ws] + [wseg])
    njobs = ops.repack_stale()
    assert njobs == sum(len(ws) for ws, _, _ in expect) + 1 and L.launches - n0 == 1
    for ws, cfg, tr in expect:
        cin, st = ws[0].shape[1], cfg.stride
        ref = torch.zeros_like(ops.packed_weights(tuple(ws), cfg, tr))
        off = 0
        for w in ws:
            L.call("s2e_pack_weight", L.ptr(w), w.shape[0], cin, cfg.kh, cfg.kw, st, cfg.pad, int(tr), sum(x.shape[0] for x in ws),
                   off, cfg.cin_pad, L.ptr(ref), L.stream())
            off += w.shape[0]
        assert torch.equal(ops.packed_weights(tuple(ws), cfg, tr), ref)
    ops._pack_cache.clear()


def test_adam_multi_matches_torch(S):
    L, ops = S
    from seg2eye_b200 import optim
    g = torch.Generator().manual_seed(9)
    shapes = [(5,), (4096,), (4097,), (3, 1000, 3), (130, 72, 3, 3), (1,)] + [(17 + i,) for i in range(60)]
    p0 = [torch.randn(*s, generator=g) for s in shapes]
    pr = [p.clone().requires_grad_() for p in p0]
    pc = [p.cuda().requires_grad_() for p in p0]
    o_r = torch.optim.Adam(pr, lr=2e-3, betas=(0.0, 0.9), weight_decay=0.01)
    o_c = optim.Adam(pc, lr=2e-3, betas=(0, 0.9), weight_decay=0.01)
    for it in range(3):
        for a, b in zip(pr, pc):
            gr = torch.randn(a.shape, generator=g)
            a.grad, b.grad = gr.clone(), gr.cuda()
        pc[3].grad = pr[3].grad = None      # a parameter that never receives a gradient (fc_var) is skipped, like torch does
        n0 = L.launches
        o_r.step()
        o_c.step()
        assert L.launches - n0 <= 4    # prepare + ceil(66/48) multi launches (+ no re-pack: nothing registered)
    for a, b in zip(pr, pc):
        assert rel(b, a) < 1e-6
    assert torch.equal(pc[3].detach().cpu(), p0[3])


def test_spectral_batch_matches_torch(S):
    """Several layers x several successive calls in one batched call == torch's power iteration applied call by call."""
    L, ops = S
    g = torch.Generator().manual_seed(4)
    shapes = [(64, 1, 3, 3), (48, 20, 3, 3), (130, 64, 4, 4), (256, 129, 1, 1)]
    layers, refs = [], []
    for s in shapes:
        w = torch.randn(*s, generator=g)
        u = F.normalize(torch.randn(s[0], generator=g), dim=0)
        v = F.normalize(torch.randn(w[0].numel(), generator=g), dim=0)
        layers.append((w.cuda(), u.cuda(), v.cuda()))
        refs.append((w.view(s[0], -1), u, v))
    n_calls = 3
    out = ops.spectral_batch(layers, True, n_calls, keep_uv=True)
    for (inv, U, V), (wm, u, v), (wc, uc, vc) in zip(out, refs, layers):
        for c in range(n_calls):
            v = F.normalize(torch.mv(wm.t(), u), dim=0, eps=1e-12)
            u = F.normalize(torch.mv(wm, v), dim=0, eps=1e-12)
            sigma = torch.dot(u, torch.mv(wm, v))
            assert rel(U[c], u) < 2e-5 and rel(V[c], v) < 2e-5 and abs(float(inv[c]) * float(sigma) - 1) < 2e-5
        assert rel(uc, u) < 2e-5 and rel(vc, v) < 2e-5
    # batched == one layer at a time, bit for bit (grouping layers into a table does not change the arithmetic)
    l2 = [(w.clone(), F.normalize(torch.ones_like(u), dim=0), F.normalize(torch.ones_like(v), dim=0)) for w, u, v in layers]
    l3 = [(w.clone(), u.clone(), v.clone()) for w, u, v in l2]
    a = ops.spectral_batch(l2, True)
    b = [ops.spectral_batch([l], True)[0] for l in l3]
    for (ia, _, _), (ib, _, _), x, y in zip(a, b, l2, l3):
        assert torch.equal(ia, ib) and torch.equal(x[1], y[1]) and torch.equal(x[2], y[2])
    # eval mode leaves the buffers alone
    before = [(u.clone(), v.clone()) for _, u, v in layers]
    ev = ops.spectral_batch(layers, False, 2, keep_uv=True)
    for (inv, U, V), (w, u, v), (u0, v0) in zip(ev, layers, before):
        assert torch.equal(u, u0) and torch.equal(v, v0) and torch.equal(U[1], u0) and float(inv[0]) == float(inv[1])
        wm = w.view(w.shape[0], -1)
        assert abs(float(inv[0]) * float(torch.dot(u, torch.mv(wm, v))) - 1) < 2e-5


# ------------------------------------------------------------------------------------------ fused residual / padded head
@pytest.mark.parametrize("impl_name,Cout", [("tc", 128), ("tc", 64), ("tc", 72), ("simt", 64)])
def test_conv_residual_in_epilogue(S, impl_name, Cout):
    """x_s + conv_1(h) (architecture.py:44): the residual rides in the tcgen05 epilogue (Cout % 64 == 0) or is added by
    the add kernel (other shapes / SIMT); either way one op, same gradients (d res = dy)."""
    L, ops = S
    g = torch.Generator().manual_seed(21)
    B, Cin, H, W = 2, 64, 21, 17
    x = bf(torch.randn(B, Cin, H, W, generator=g))
    w = bf(torch.randn(Cout, Cin, 3, 3, generator=g) / (Cin * 9) ** 0.5)
    b = torch.randn(Cout, generator=g) * 0.1
    r = bf(torch.randn(B, Cout, H, W, generator=g))
    xr, wr, br, rr = [t.clone().requires_grad_() for t in (x, w, b, r)]
    yr = F.conv2d(xr, wr * 0.8, br, padding=1) + rr
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc, rc = nhwc(x).requires_grad_(), nhwc(r).requires_grad_()
    wc, bc = w.cuda().requires_grad_(), b.cuda().requires_grad_()
    u = F.normalize(torch.randn(Cout, generator=g), dim=0).cuda()
    v = F.normalize(torch.randn(Cin * 9, generator=g), dim=0).cuda()
    with ops.force_impl(L.IMPL_TC if impl_name == "tc" else L.IMPL_SIMT):
        y = ops.tap_conv(xc, ops.ConvCfg(3, 3, 1, 1, L.ACT_NONE), (wc,), (bc,), (u, v, torch.tensor([0.8], device="cuda")), rc)
        y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < 5e-3
    assert torch.equal(nchw(rc.grad), dy)
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT and rel(bc.grad, br.grad) < TOL_ACT


@pytest.mark.parametrize("case", [(3, 128, 11, 9, 4, 2), (2, 512, 33, 18, 4, 2), (1, 1024, 9, 7, 4, 2), (2, 192, 20, 16, 3, 1),
                                  (2, 256, 5, 40, 4, 2)])
def test_head_conv_tap_channel_form(S, case):
    """PatchGAN logit head (discriminator.py:38) as D[q][t] = x[q] . W[t] + gather (ops.HeadConvFn): forward, data gradient,
    weight and bias gradient vs torch; the layer module picks this route for a (1, Cin, k, k) weight."""
    L, ops = S
    B, Cin, H, W, k, pad = case
    g = torch.Generator().manual_seed(31)
    x = bf(torch.randn(B, Cin, H, W, generator=g))
    w = bf(torch.randn(1, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5)
    b = torch.randn(1, generator=g) * 0.1
    xr, wr, br = [t.clone().requires_grad_() for t in (x, w, b)]
    yr = F.conv2d(xr, wr, br, padding=pad)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    from seg2eye_b200.models.networks.layers import Conv2d
    conv = Conv2d(Cin, 1, k, stride=1, padding=pad).cuda()
    with torch.no_grad():
        conv.weight.copy_(w)
        conv.bias.copy_(b)
    xc = nhwc(x).requires_grad_()
    assert ops.head_conv_ok(xc, conv.cfg, conv.weight)
    y = conv.forward_nhwc(xc)
    assert y.grad_fn.name().startswith("HeadConvFn")
    y.backward(nhwc(dy))
    assert rel(nchw(y), yr) < 5e-3, rel(nchw(y), yr)             # fp32 dot products, one bf16 rounding on the logit
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT, rel(nchw(xc.grad), xr.grad)
    assert rel(conv.weight.grad, wr.grad) < TOL_ACT, rel(conv.weight.grad, wr.grad)
    assert rel(conv.bias.grad, br.grad) < TOL_ACT
    # a second call after a weight update sees the new weight (packed copy and the [Cin][64] data-gradient copy refresh)
    with torch.no_grad():
        conv.weight.mul_(-0.5)
    xc.grad = None
    y2 = conv.forward_nhwc(xc)
    y2.backward(nhwc(dy))
    assert rel(nchw(y2) - b.view(1, 1, 1, 1), -0.5 * (yr.detach() - b.view(1, 1, 1, 1))) < 1e-2
    assert rel(nchw(xc.grad), -0.5 * xr.grad) < TOL_ACT


@pytest.mark.parametrize("mode", ["hinge", "w"])
def test_gan_loss_sums_fused_into_the_logit_head(S, mode):
    """The discriminator's logit head reduces, in its gather kernel, the sums behind GANLoss's hinge / Wasserstein terms
    (loss.py:58-83) for both halves of a [fake ; real] batch; Pix2PixModel.divide_pred tags the halves and GANLoss then skips its
    own reduction.  Values and gradients must equal the separate reduction kernels' (same bf16 logits, fp32 sums)."""
    L, ops = S
    from seg2eye_b200.models.networks.layers import Conv2d
    from seg2eye_b200.models.networks.loss import GANLoss
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    g = torch.Generator().manual_seed(17)
    conv = Conv2d(128, 1, 4, stride=1, padding=2).cuda()
    x = nhwc(bf(torch.randn(6, 128, 13, 11, generator=g) * 3)).requires_grad_()
    crit = GANLoss(mode)
    cases = [(0, True, False), (0, False, True), (1, True, True)]    # (half, target_is_real, for_discriminator)
    res = {}
    for fused in (True, False):
        y = conv.forward_nhwc(x)
        assert hasattr(y, "_s2e_gan_sums")
        if not fused:
            del y._s2e_gan_sums
        halves = Pix2PixModel.divide_pred(None, y)
        assert hasattr(halves[0], "_s2e_gan_half") == fused
        hits0 = ops._state.get("gan_presummed", 0)
        losses = [crit(halves[h], real, for_discriminator=ford) for h, real, ford in cases]
        assert ops._state.get("gan_presummed", 0) - hits0 == (3 if fused else 0)
        x.grad = None
        sum(losses).backward()
        res[fused] = ([float(l.detach()) for l in losses], x.grad.float().clone())
    for a, b in zip(res[True][0], res[False][0]):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(b)), (res[True][0], res[False][0])
    assert rel(res[True][1].cpu(), res[False][1].cpu()) < 1e-6
    ref = nchw(conv.forward_nhwc(x).detach())
    want = {("hinge", 0): -float(ref[:3].mean()), ("w", 0): -float(ref[:3].mean()),
            ("hinge", 1): -float(torch.clamp(-ref[:3] - 1, max=0).mean()), ("w", 1): float(ref[:3].mean()),
            ("hinge", 2): -float(torch.clamp(ref[3:] - 1, max=0).mean()), ("w", 2): -float(ref[3:].mean())}
    for i in range(3):
        assert abs(res[True][0][i] - want[(mode, i)]) < 1e-4 * max(1.0, abs(want[(mode, i)])), (i, res[True][0], want)


def test_one_channel_head_on_tensor_cores(S):
    """PatchGAN logit head (512 -> 1, 4x4 s1 p2; discriminator.py:96) with cout_pad: zero-padded output channels on the
    tcgen05 kernels; forward, data gradient, weight and bias gradient vs torch."""
    L, ops = S
    g = torch.Generator().manual_seed(22)
    B, Cin, H, W = 3, 128, 11, 9
    x = bf(torch.randn(B, Cin, H, W, generator=g))
    w = bf(torch.randn(1, Cin, 4, 4, generator=g) / (Cin * 16) ** 0.5)
    b = torch.randn(1, generator=g) * 0.1
    xr, wr, br = [t.clone().requires_grad_() for t in (x, w, b)]
    yr = F.conv2d(xr, wr, br, padding=2)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc, wc, bc = nhwc(x).requires_grad_(), w.cuda().requires_grad_(), b.cuda().requires_grad_()
    from seg2eye_b200 import ops as O2
    O2.profile_begin()
    y = ops.tap_conv(xc, ops.ConvCfg(4, 4, 1, 2, L.ACT_NONE, False, 0, 64), (wc,), (bc,))
    assert y.shape == (B, H + 1, W + 1, 1)
    y.backward(nhwc(dy))
    prof = O2.profile_end()
    assert prof["tc_n"] == 3      # forward, data gradient and weight gradient all ran on the tcgen05 kernels
    assert rel(nchw(y), yr) < TOL_ACT
    assert rel(nchw(xc.grad), xr.grad) < TOL_ACT
    assert rel(wc.grad, wr.grad) < TOL_ACT and rel(bc.grad, br.grad) < TOL_ACT
    # the layer itself takes the tap-channel head route (test_head_conv_tap_channel_form)
    from seg2eye_b200.models.networks.layers import Conv2d
    conv = Conv2d(512, 1, 4, stride=1, padding=2).cuda()
    x2 = bf(torch.randn(2, 512, 6, 5, generator=g))
    y2 = conv.forward_nhwc(nhwc(x2))
    ref = F.conv2d(x2, bf(conv.weight.detach().cpu()), conv.bias.detach().cpu(), padding=2)
    assert y2.shape == (2, 7, 6, 1) and rel(nchw(y2), ref) < TOL_ACT


@pytest.mark.parametrize("act,C", [(1, 64), (0, 128)])
def test_spade_style_on_upsampled_input_without_materialising_it(S, act, C):
    """SpadeStyleFn(up=True) on x == SpadeStyleFn on nearest-2x(x) (generator.py:50 + normalization.py:91-105), forward,
    running statistics and all gradients; two consumers of the same x share one gradient buffer (GradSink)."""
    L, ops = S
    g = torch.Generator().manual_seed(12)
    B, h, w = 2, 6, 5
    x = bf(torch.randn(B, C, h, w, generator=g) + 0.2)
    gam = [bf(torch.randn(B, C, 2 * h, 2 * w, generator=g) * 0.5) for _ in range(2)]
    bet = [bf(torch.randn(B, C, 2 * h, 2 * w, generator=g) * 0.5) for _ in range(2)]
    style = [torch.randn(B, 2 * C, generator=g) * 0.5 for _ in range(2)]
    dout = [bf(torch.randn(B, C, 2 * h, 2 * w, generator=g)) for _ in range(2)]
    acts = (act, 0)
    # reference: materialised up-sampling, two SPADE+Style blocks on it (like norm_0 / norm_s)
    xr = x.clone().requires_grad_()
    grs, brs, srs = [t.clone().requires_grad_() for t in gam], [t.clone().requires_grad_() for t in bet], [t.clone().requires_grad_() for t in style]
    xu = F.interpolate(xr, scale_factor=2, mode="nearest")
    rms, rvs, refs, tot = [], [], [], 0
    for i in range(2):
        rm, rv = torch.zeros(C), torch.ones(C)
        xn = F.batch_norm(xu, rm, rv, training=True, momentum=0.1, eps=1e-5)
        o = 0.5 * (xn * (1 + grs[i]) + brs[i] + xu * (1 + srs[i][:, :C, None, None]) + srs[i][:, C:, None, None])
        if acts[i]:
            o = F.leaky_relu(o, 0.2)
        tot = tot + (o * dout[i]).sum()
        rms.append(rm), rvs.append(rv), refs.append(o.detach())
    tot.backward()
    # ours
    xc0 = nhwc(x).requires_grad_()
    xc = ops.AddFn.apply(xc0, torch.zeros_like(xc0))
    sink = ops.GradSink()
    outs, gbs, scs, bufs = [], [], [], []
    for i in range(2):
        gbc = torch.cat([nhwc(gam[i]), nhwc(bet[i])], dim=3).contiguous().requires_grad_()
        sc = style[i].cuda().requires_grad_()
        rmc, rvc, nbt = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda"), torch.tensor(0, device="cuda")
        cfg = ops.NormCfg(False, acts[i], True, 0.1, 1e-5)
        outs.append(ops.SpadeStyleFn.apply(xc, gbc, sc, cfg, rmc, rvc, nbt, True, sink))
        gbs.append(gbc), scs.append(sc), bufs.append((rmc, rvc))
    assert outs[0].shape == (B, 2 * h, 2 * w, C)
    sum((o.float() * nhwc(d).float()).sum() for o, d in zip(outs, dout)).backward()
    for i in range(2):
        assert rel(nchw(outs[i]), refs[i]) < 5e-3
    assert rel(nchw(xc0.grad), xr.grad) < TOL_ACT
    for i in range(2):
        assert rel(nchw(gbs[i].grad[..., :C]), grs[i].grad) < TOL_ACT and rel(nchw(gbs[i].grad[..., C:]), brs[i].grad) < TOL_ACT
        assert rel(scs[i].grad, srs[i].grad) < TOL_ACT
        assert rel(bufs[i][0], rms[i]) < 1e-4 and rel(bufs[i][1], rvs[i]) < 1e-4
    assert sink.buf is None and sink.seen == 0


@pytest.mark.parametrize("B,H,W", [(2, 21, 37), (1, 45, 150), (3, 8, 128), (1, 7, 300)])
def test_conv_img_with_fused_leaky_relu_input(S, B, H, W):
    """leaky_relu(x, 0.2) -> conv 64->1 3x3 (generator.py:97-98) as ONE forward kernel; its backward applies the
    LeakyReLU derivative inside the data-gradient kernel and the activation inside the weight-gradient kernel."""
    L, ops = S
    from seg2eye_b200.models.networks.layers import Conv2d
    g = torch.Generator().manual_seed(31)
    x = bf(torch.randn(B, 64, H, W, generator=g))
    conv = Conv2d(64, 1, 3, padding=1).cuda()
    w = bf(conv.weight.detach().cpu())
    conv.weight.data.copy_(w)
    xr, wr, br = x.clone().requires_grad_(), w.clone().requires_grad_(), conv.bias.detach().cpu().clone().requires_grad_()
    yr = F.conv2d(F.leaky_relu(xr, 0.2), wr, br, padding=1)
    dy = bf(torch.randn(yr.shape, generator=g))
    yr.backward(dy)
    xc = nhwc(x).requires_grad_()
    n0 = L.launches
    y = conv.forward_nhwc(xc, in_act=L.ACT_LRELU)
    assert L.launches - n0 <= 2          # (weight pack +) one convolution kernel: no separate activation pass
    y.backward(nhwc(dy))
    # mma.sync kernels with fp32 accumulation: only the bf16 rounding of the outputs is left
    assert rel(nchw(y), yr) < 4e-3, rel(nchw(y), yr)
    assert rel(nchw(xc.grad), xr.grad) < 4e-3, rel(nchw(xc.grad), xr.grad)
    assert rel(conv.weight.grad, wr.grad) < 2e-3 and rel(conv.bias.grad, br.grad) < TOL_ACT, rel(conv.weight.grad, wr.grad)
    # other shapes fall back to the separate activation kernel with identical results
    conv2 = Conv2d(16, 1, 3, padding=1).cuda()
    x2 = bf(torch.randn(B, 16, H, W, generator=g))
    ref2 = F.conv2d(F.leaky_relu(x2, 0.2), bf(conv2.weight.detach().cpu()), conv2.bias.detach().cpu(), padding=1)
    assert rel(nchw(conv2.forward_nhwc(nhwc(x2), in_act=L.ACT_LRELU)), ref2) < TOL_ACT


@pytest.mark.parametrize("C,up,act,per_sample", [(64, False, 1, False), (128, True, 1, False), (128, False, 0, True), (64, True, 0, False)])
def test_spade_modulation_fused_into_gamma_beta_conv(S, C, up, act, per_sample):
    """No-grad SPADE+Style block with gamma|beta consumed in the epilogue of their own convolution
    (ops.spade_conv_fused) == convolution followed by the modulation kernel == the fp32 statement of
    normalization.py:91-105,161-192; BatchNorm running buffers advance identically."""
    L, ops = S
    g = torch.Generator().manual_seed(41)
    B, H, W = 3, 16, 32
    hx, wx = (H // 2, W // 2) if up else (H, W)
    x = bf(torch.randn(B, C, hx, wx, generator=g) * 1.3 + 0.2)
    actv = bf(torch.relu(torch.randn(B, 128, H, W, generator=g)))
    wg = bf(torch.randn(C, 128, 3, 3, generator=g) / 34.0)
    wb = bf(torch.randn(C, 128, 3, 3, generator=g) / 34.0)
    bg, bb = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    style = torch.randn(B, 2 * C, generator=g) * 0.5
    # fp32 reference
    xu = F.interpolate(x, scale_factor=2, mode="nearest") if up else x
    gam, bet = F.conv2d(actv, wg, bg, padding=1), F.conv2d(actv, wb, bb, padding=1)
    rm, rv = torch.zeros(C), torch.ones(C)
    xn = F.instance_norm(xu, eps=1e-5) if per_sample else F.batch_norm(xu, rm, rv, training=True, momentum=0.1, eps=1e-5)
    ref = 0.5 * (xn * (1 + gam) + bet + xu * (1 + style[:, :C, None, None]) + style[:, C:, None, None])
    if act:
        ref = F.leaky_relu(ref, 0.2)
    cfg = ops.NormCfg(per_sample, act, True, 0.1, 1e-5)
    ccfg = ops.ConvCfg(3, 3, 1, 1, L.ACT_NONE)
    ws, bs = (wg.cuda(), wb.cuda()), (bg.cuda(), bb.cuda())
    outs = []
    with torch.no_grad():
        assert ops.spade_conv_fused_ok(nhwc(x), up, 128)
        for fused in (True, False):
            rmc, rvc, nbt = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda"), torch.tensor(0, device="cuda")
            bufs = (None, None, None) if per_sample else (rmc, rvc, nbt)
            if fused:
                o = ops.spade_conv_fused(nhwc(actv), ccfg, ws, bs, nhwc(x), style.cuda(), cfg, *bufs, up)
            else:
                gb = ops.tap_conv(nhwc(actv), ccfg, ws, bs)
                o = ops.SpadeStyleFn.apply(nhwc(x), gb, style.cuda(), cfg, *bufs, up)
            outs.append(o)
            if not per_sample:
                assert rel(rmc, rm) < 1e-4 and rel(rvc, rv) < 1e-4 and int(nbt) == 1
    assert outs[0].shape == (B, H, W, C)
    assert rel(nchw(outs[0]), ref) < 5e-3 and rel(nchw(outs[1]), ref) < TOL_ACT
    assert rel(outs[0], outs[1]) < TOL_ACT


@pytest.mark.parametrize("C,up,act", [(64, False, 1), (128, True, 1), (128, False, 0)])
def test_spade_conv_fused_training_forward_backward(S, C, up, act):
    """SpadeConvFn (gamma|beta convolution + modulation in one kernel, gamma and the activation mask kept for backward)
    against fp32 autograd through conv2d + batch_norm + the modulation formula: output, running buffers and the
    gradients w.r.t. actv, x, style, both weights and both biases."""
    L, ops = S
    g = torch.Generator().manual_seed(43)
    B, H, W = 2, 16, 32
    hx, wx = (H // 2, W // 2) if up else (H, W)
    x = bf(torch.randn(B, C, hx, wx, generator=g) * 1.3 + 0.2)
    actv = bf(torch.relu(torch.randn(B, 128, H, W, generator=g)))
    wg = bf(torch.randn(C, 128, 3, 3, generator=g) / 34.0)
    wb = bf(torch.randn(C, 128, 3, 3, generator=g) / 34.0)
    bg, bb = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    style = torch.randn(B, 2 * C, generator=g) * 0.5
    dout = bf(torch.randn(B, C, H, W, generator=g))
    ref_in = [t.clone().requires_grad_() for t in (actv, x, style, wg, wb, bg, bb)]
    ar, xr, sr, wgr, wbr, bgr, bbr = ref_in
    xu = F.interpolate(xr, scale_factor=2, mode="nearest") if up else xr
    gam, bet = F.conv2d(ar, wgr, bgr, padding=1), F.conv2d(ar, wbr, bbr, padding=1)
    rm, rv = torch.zeros(C), torch.ones(C)
    xn = F.batch_norm(xu, rm, rv, training=True, momentum=0.1, eps=1e-5)
    ref = 0.5 * (xn * (1 + gam) + bet + xu * (1 + sr[:, :C, None, None]) + sr[:, C:, None, None])
    if act:
        ref = F.leaky_relu(ref, 0.2)
    ref.backward(dout)
    ac, xc = nhwc(actv).requires_grad_(), nhwc(x).requires_grad_()
    sc = style.cuda().requires_grad_()
    wgc, wbc, bgc, bbc = [t.cuda().requires_grad_() for t in (wg, wb, bg, bb)]
    rmc, rvc, nbt = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda"), torch.tensor(0, device="cuda")
    cfg = ops.NormCfg(False, act, True, 0.1, 1e-5)
    out = ops.SpadeConvFn.apply(ac, xc, sc, wgc, wbc, bgc, bbc, ops.ConvCfg(3, 3, 1, 1, L.ACT_NONE), cfg, rmc, rvc, nbt, up, None)
    out.backward(nhwc(dout))
    assert rel(nchw(out), ref) < 5e-3
    assert rel(rmc, rm) < 1e-4 and rel(rvc, rv) < 1e-4 and int(nbt) == 1
    assert rel(nchw(ac.grad), ar.grad) < TOL_ACT and rel(nchw(xc.grad), xr.grad) < TOL_ACT
    assert rel(sc.grad, sr.grad) < TOL_ACT
    assert rel(wgc.grad, wgr.grad) < TOL_ACT and rel(wbc.grad, wbr.grad) < TOL_ACT
    assert rel(bgc.grad, bgr.grad) < TOL_ACT and rel(bbc.grad, bbr.grad) < TOL_ACT


# ------------------------------------------------------------------------------------------ forward kernel variants
@pytest.mark.parametrize("key6", [8, 4, 12])
def test_conv_tcgen05_forward_kernel_variants(S, key6):
    """Layers with Cout <= 128 run with swapped MMA operands by default (weights = A, two pixel sub-tiles = one N = 256 operand,
    transposed epilogue), and small maps take single 128-pixel tiles.  Debug key 6 bit 3 keeps the pixels on the M side (the
    N = 64 / 128 kernels these layers used before, still used by the fused SPADE epilogues), bit 2 forces double tiles: all
    combinations must agree with torch, on the plain cases and on the mask / residual / fused-SPADE epilogues."""
    L, ops = S
    L.call("s2e_debug_set", 6, key6)
    L.call("s2e_debug_set", 5, 2 if key6 & 8 else 0)     # with bit 3 also the weight-gradient kernels without merged taps
    try:
        for case in [TC_CASES[0], TC_CASES[1], TC_CASES[3], TC_CASES[4], TC_CASES[5], TC_CASES[8], TC_CASES[10], TC_CASES[11],
                     (1, 64, 64, 37, 29, 3, 1, 1, 0), (3, 128, 128, 40, 48, 3, 1, 1, 2)]:
            conv_case(S, L.IMPL_TC, *case)
        test_conv_residual_in_epilogue(S, "tc", 128)
        test_conv_residual_in_epilogue(S, "tc", 64)
        test_relu_backward_fused_into_dgrad_epilogue(S, "tc")
        test_spade_modulation_fused_into_gamma_beta_conv(S, 64, False, 1, False)
        test_spade_conv_fused_training_forward_backward(S, 64, False, 1)
    finally:
        L.call("s2e_debug_set", 6, 0)
        L.call("s2e_debug_set", 5, 0)


# ------------------------------------------------------------------------------------------ halo-tile forward kernel
HALO_CASES = [
    (2, 128, 128, 24, 16, 3, 1, 1, 0),     # N = 128, two sub-tiles
    (1, 64, 64, 20, 16, 3, 1, 1, 0),       # N = 64, partial tile at the bottom (H = 20)
    (1, 256, 128, 40, 32, 3, 1, 1, 1),     # four 64-channel blocks, fused LeakyReLU
    (2, 128, 64, 24, 16, 3, 1, 1, 0),
    (1, 64, 64, 37, 29, 3, 1, 1, 0),       # ragged: partial tiles right and bottom, odd tile count
    (3, 128, 128, 40, 48, 3, 1, 1, 0),     # 54 halo tiles in 27 work items: one per CTA (test_gpu_conv_exact.py loops)
    (1, 64, 72, 16, 8, 3, 1, 1, 1),        # Cout not a multiple of 64
    (2, 64, 256, 24, 16, 3, 1, 1, 0),      # forward N = 256 (plain kernel), data gradient N = 64 (halo kernel)
]


@pytest.mark.parametrize("case", HALO_CASES)
def test_conv_tcgen05_halo_kernel(S, case):
    """3x3 / stride-1 convolutions with an N tile <= 128 through the halo-tile kernel (one staged {64, 10, 18} input tile
    per 64-channel block serves all nine taps via UMMA descriptors on shifted windows): forward and data gradient."""
    L, ops = S
    ops.set_halo(True)
    try:
        conv_case(S, L.IMPL_TC, *case)
    finally:
        ops.set_halo(False)


def test_halo_kernel_epilogue_variants(S):
    """Residual add, fused ReLU-backward mask and the fused SPADE+Style epilogues (no-grad and training) on the halo kernel."""
    L, ops = S
    ops.set_halo(True)
    try:
        test_conv_residual_in_epilogue(S, "tc", 128)
        test_conv_residual_in_epilogue(S, "tc", 64)
        test_relu_backward_fused_into_dgrad_epilogue(S, "tc")
        test_spade_modulation_fused_into_gamma_beta_conv(S, 64, False, 1, False)
        test_spade_modulation_fused_into_gamma_beta_conv(S, 64, True, 0, False)
        test_spade_conv_fused_training_forward_backward(S, 64, False, 1)
    finally:
        ops.set_halo(False)
