"""Bit-exact tests of the tcgen05 convolutions with integer-valued inputs.

Activations and output gradients take values in {-1, 0, 1}, weights are sparse in {-1, 0, 1} and biases are small
integers, with at most 256 - |bias| non-zero weights per output channel and at most 256 per input channel.  Every partial
sum is then an integer far below 2^24, so neither the summation order nor the fp32 accumulation (TMEM, split-K atomics)
can change a result: every forward and data-gradient output is an integer with |v| <= 256 (exact in bf16) and every
weight gradient an exact fp32 integer.  The kernels must therefore match a float64 reference bit for bit, and one
missing, duplicated or misplaced product moves some output by at least 1.  Where the product path rounds (LeakyReLU in
fp32 before the bf16 store, a LeakyReLU backward that hands bf16 multiples of 0.2 to the data gradient) the reference
rounds at the same place, so each result is still one exact value rounded once.

The persistent-regime cases launch at least three work items per CTA on every forward kernel instantiation the
benchmarked training step uses, so both TMEM accumulator slots, the accumulator phase flip and the reuse of the output
staging buffers are exercised; each case asserts that bound for the device it runs on.  A mismatch is reported with the
(b, h, w, c) of the first wrong element, the number of wrong elements, and the pixel tile, work item, CTA and loop
iteration of the forward kernel that wrote it (from a mirror of the host's tile rule, `fwd_launch`)."""
import contextlib
import zlib

import pytest
import torch
import torch.nn.functional as F

from test_gpu_kernels import HALO_CASES, MT_WGRAD_CASES, TC_CASES

B200_SMS = 148
BM = 128                     # pixels per sub-tile of the forward kernels
U32 = 2.0 ** -24             # unit roundoff of fp32
BF16_ULP_REL = 2.0 ** -8     # one bf16 ulp relative to the magnitude of the value (8 significant bits)
ACT_NONE, ACT_LRELU, ACT_RELU = 0, 1, 2
LRELU_SLOPE = torch.tensor(0.2, dtype=torch.float32)    # the kernels multiply by 0.2f


def ceil_div(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------ launch geometry (host mirror)
def choose_fwd_tile(B, H, W):
    """Mirror of choose_fwd_tile (csrc/conv_tc.cu): the pixel tile (w, h, b) of <= 128 pixels with the fewest tiles."""
    best, pick = None, (1, 1, 1)
    for w in range(1, min(W, BM) + 1):
        for h in range(1, H + 1):
            if w * h > BM:
                break
            b = max(1, min(B, BM // (w * h)))
            score = ceil_div(W, w) * ceil_div(H, h) * ceil_div(B, b) * 1024 - w
            if best is None or score < best:
                best, pick = score, (w, h, b)
    return pick


def fwd_launch(B, Ho, Wo, Cout, Cin, ntaps, side=False, spade=False, halo=False, tile=None, sms=B200_SMS):
    """Geometry of one s2e_tapconv_fwd launch on the tcgen05 path (mirror of s2e_tapconv_fwd_tc and launch_fwd):
    N tile, 128-pixel sub-tiles per work item, pixel tile, work items and grid.  `side`: a ReLU mask or a residual."""
    if spade:
        bn = Cout
    elif Cout >= 256:
        bn = 256
    elif not halo and Cout >= 64 and (Cout >= 128 or (ntaps * Cin >= 512 and not side)):
        bn = 128                 # swapped operands (MODE 3)
    else:
        bn = 128 if Cout >= 128 else 64
    mt_max = 1 if bn == 256 else 2
    tw, th, tb = (8, 16, 1) if halo else (tile or choose_fwd_tile(B, Ho, Wo))
    g = dict(bn=bn, tw=tw, th=th, tb=tb, tiles_w=ceil_div(Wo, tw), tiles_h=ceil_div(Ho, th), tiles_b=ceil_div(B, tb),
             tiles_n=ceil_div(Cout, bn), mt=mt_max)
    g["tiles_m"] = g["tiles_w"] * g["tiles_h"] * g["tiles_b"]
    if not halo and not spade and mt_max == 2:
        w1 = ceil_div(g["tiles_m"] * g["tiles_n"], sms) * 6
        w2 = ceil_div(ceil_div(g["tiles_m"], 2) * g["tiles_n"], sms) * 10
        if w1 < w2:
            g["mt"] = 1
    g["items"] = ceil_div(g["tiles_m"], g["mt"]) * g["tiles_n"]
    g["grid"] = min(g["items"], sms)
    return g


def work_items_lower_bound(B, Ho, Wo, Cout):
    """Work items of a forward launch whatever pixel tile and kernel are picked: a tile holds at most 128 pixels, a work
    item at most 2 sub-tiles (1 on the N = 256 kernel) and the N tile is at most 256 (128 for Cout <= 128)."""
    mt, bn = (1, 256) if Cout >= 256 else (2, 128)
    return ceil_div(B * Ho * Wo, BM * mt) * ceil_div(Cout, bn)


def locate(g, b, h, w, c):
    """Tile, work item, CTA and loop iteration of the forward kernel that writes output element (b, h, w, c)."""
    m = ((b // g["tb"]) * g["tiles_h"] + h // g["th"]) * g["tiles_w"] + w // g["tw"]
    item = (m // g["mt"]) * g["tiles_n"] + c // g["bn"]
    return "pixel tile %d (sub-tile %d of work item %d of %d), CTA %d, iteration %d of its loop" % (
        m, m % g["mt"], item, g["items"], item % g["grid"], item // g["grid"])


# ------------------------------------------------------------------------------------------ integer-valued inputs
def ternary(shape, gen, density=2.0 / 3.0, nonneg=False):
    """Values in {-1, 0, 1} ({0, 1} with nonneg), non-zero with probability `density`."""
    nz = torch.rand(shape, generator=gen) < density
    sign = torch.ones(shape) if nonneg else torch.randint(0, 2, shape, generator=gen).float() * 2 - 1
    return sign * nz


def int_bias(n, gen, mag=3):
    return torch.randint(-mag, mag + 1, (n,), generator=gen).float()


def sparse_weight(Cout, Cin, kh, kw, gen, bias=None, extra=0, cin_live=None, target=160):
    """Sparse {-1, 0, 1} OIHW weight.  Output channel o keeps at most 256 - |bias[o]| - extra non-zeros over its
    K = kh*kw*Cin (extra: a residual adds one more unit), input channel i at most 256 over kh*kw*Cout (data gradient).
    cin_live: only the first cin_live input channels are non-zero (channel-padded layers)."""
    cin_live = Cin if cin_live is None else cin_live
    taps = kh * kw
    p = min(1.0, target / (taps * cin_live), target / (taps * Cout))
    w = ternary((Cout, Cin, kh, kw), gen, density=p)
    w[:, cin_live:] = 0
    row_cap = 256 - extra - (bias.abs().long() if bias is not None else torch.zeros(Cout, dtype=torch.long))
    for o in range(Cout):            # drop the surplus non-zeros (a random subset) of a row, then of a column
        nz = w[o].flatten().nonzero().flatten()
        if len(nz) > row_cap[o]:
            drop = nz[torch.randperm(len(nz), generator=gen)[:len(nz) - int(row_cap[o])]]
            w[o].view(-1)[drop] = 0
    for i in range(Cin):
        col = w[:, i].clone()
        nz = col.flatten().nonzero().flatten()
        if len(nz) > 256:
            drop = nz[torch.randperm(len(nz), generator=gen)[:len(nz) - 256]]
            col.view(-1)[drop] = 0
            w[:, i] = col
    check_weight_bounds(w, bias, extra)
    return w


def check_weight_bounds(w, bias=None, extra=0):
    """The bounds that keep every forward and data-gradient result an integer within +-256."""
    nnz = w.ne(0)
    row = nnz.sum(dim=(1, 2, 3))
    col = nnz.sum(dim=(0, 2, 3))
    b = bias.abs() if bias is not None else torch.zeros(w.shape[0])
    assert bool(w.abs().le(1).all()) and bool((w == w.round()).all())
    assert bool((row + b + extra).le(256).all()), "output channel over its non-zero budget"
    assert bool(col.le(256).all()), "input channel over its non-zero budget"
    return int(row.max()), int(col.max())


def bf16_round(t):
    """Round-to-nearest-even to bf16 (via fp32, which must hold the value exactly)."""
    t32 = t.float()
    assert torch.equal(t32.double(), t.double()), "value not exact in fp32"
    return t32.to(torch.bfloat16).float()


def act_fwd_ref(v, act):
    """act_t in fp32 (max(v, 0.2f*v) for LeakyReLU) followed by the bf16 store; v exact in fp32."""
    v32 = v.float()
    assert torch.equal(v32.double(), v.double())
    if act == ACT_LRELU:
        v32 = torch.maximum(v32, v32 * LRELU_SLOPE.to(v32.device))
    elif act == ACT_RELU:
        v32 = torch.clamp_min(v32, 0.0)
    return v32.to(torch.bfloat16).float()


def act_bwd_ref(dy, y, act):
    """s2e_act_bwd: dy * (y > 0 ? 1 : slope) in fp32, stored as bf16."""
    if act == ACT_NONE:
        return dy.float()
    slope = LRELU_SLOPE.to(y.device) if act == ACT_LRELU else torch.zeros((), device=y.device)
    return (dy.float() * torch.where(y > 0, torch.ones((), device=y.device), slope)).to(torch.bfloat16).float()


@contextlib.contextmanager
def exact_reference():
    """The float64 reference convolutions run without cuDNN (no FFT / Winograd rewrites of the sum)."""
    with torch.backends.cudnn.flags(enabled=False):
        yield


def conv_reference(x, w, b, stride, pad, act, dy, res=None, relu_in=False):
    """float64 forward and backward of act(conv(x, w) + b) [+ res] with the product path's roundings.
    x, w, b, dy, res: NCHW / OIHW float tensors on one device.  Returns y (bf16-valued), dx, dW, db, dpre."""
    xr = x.double().requires_grad_()
    wr = w.double().requires_grad_()
    br = b.double().requires_grad_() if b is not None else None
    with exact_reference():
        v = F.conv2d(xr, wr, br, stride=stride, padding=pad)
        if res is not None:
            v = v + res.double()
        y = act_fwd_ref(v.detach(), act)
        dpre = act_bwd_ref(dy, y, act)
        v.backward(dpre.double())
    dx = xr.grad
    if relu_in:                      # gradient w.r.t. the pre-ReLU tensor: masked where relu(a) = x > 0
        dx = dx * (x > 0)
    return y, bf16_round(dx), wr.grad, (br.grad if br is not None else None), dpre


# ------------------------------------------------------------------------------------------ comparison
def to_nhwc(t):
    return t.permute(0, 2, 3, 1)


def mismatch(got, ref, what, geom=None):
    """None if got == ref bit for bit (fp32 views), else a report: the first wrong (b, h, w, c) of an NHWC tensor (or index
    of a weight), the number of wrong elements, and with `geom` (fwd_launch) the tile / CTA that wrote the element."""
    got = got.detach().float()
    ref = ref.detach().to(got.device).float()
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    if torch.equal(got, ref):
        return None
    bad = (got != ref) | (torch.isnan(got) != torch.isnan(ref))
    n = int(bad.sum())
    first = tuple(int(i) for i in bad.nonzero()[0])
    msg = "%s: %d of %d elements differ; first at %s: got %r, want %r" % (
        what, n, got.numel(), first, float(got[first]), float(ref[first]))
    if geom is not None and got.dim() == 4:
        msg += "; written by " + locate(geom, *first)
    return msg


def assert_exact(pairs):
    """pairs: (got, ref, what, geom); every pair is compared before failing so that one report names every bad output."""
    errs = [m for m in (mismatch(*p) for p in pairs) if m]
    assert not errs, "\n".join(errs)


# ------------------------------------------------------------------------------------------ tap convolutions
def nhwc_dev(t, C=None):
    """NCHW float -> NHWC bf16 on the GPU (zero-padded to C channels)."""
    if C is not None and C > t.shape[1]:
        t = F.pad(t, (0, 0, 0, 0, 0, C - t.shape[1]))
    return to_nhwc(t).contiguous().to(torch.bfloat16).cuda()


def tap_geometries(B, Cin, Cout, H, W, k, stride, pad, cpad=0, residual=False, relu_in=False, halo=False, sms=B200_SMS):
    """fwd_launch of the forward and of the data-gradient launch of one tap convolution (None where it leaves tcgen05)."""
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    cin = max(Cin, cpad)
    if stride == 2:
        ntaps, cinp, hs, ws = ceil_div(k, 2) ** 2, 4 * cin, (H + 1) // 2, (W + 1) // 2
    else:
        ntaps, cinp, hs, ws = k * k, cin, H, W
    halo_f = halo and k == 3 and stride == 1 and Wo >= 8 and Ho >= 16 and (Ho, Wo) == (H, W)
    fwd = fwd_launch(B, Ho, Wo, Cout, cinp, ntaps, side=residual, halo=halo_f, sms=sms) \
        if cinp % 64 == 0 and Cout % 8 == 0 else None
    dgrad = fwd_launch(B, hs, ws, cinp, Cout, ntaps, side=relu_in, halo=halo_f, sms=sms) \
        if Cout % 64 == 0 and cinp % 8 == 0 else None
    return fwd, dgrad, (Ho, Wo)


def run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act=ACT_NONE, cpad=0, residual=False, relu_in=False, seed=0,
                 halo=False, min_items=0):
    """Forward, data gradient, weight and bias gradient (and the residual's gradient) of ops.tap_conv on the tcgen05 path,
    compared bit for bit with the float64 reference.  min_items: assert that many work items on the forward launch (and
    on the data-gradient launch of the same pixel count)."""
    L, ops = S
    gen = torch.Generator().manual_seed(seed)
    x = ternary((B, Cin, H, W), gen, nonneg=relu_in)
    bias = int_bias(Cout, gen)
    w = sparse_weight(Cout, Cin, k, k, gen, bias, extra=int(residual))
    fwd, dgrad, (Ho, Wo) = tap_geometries(B, Cin, Cout, H, W, k, stride, pad, cpad, residual, relu_in, halo,
                                          torch.cuda.get_device_properties(0).multi_processor_count)
    if min_items:
        assert fwd["items"] >= min_items and work_items_lower_bound(B, Ho, Wo, Cout) >= min_items, (fwd, min_items)
        if relu_in:                  # the case is there for its masked data-gradient launch
            assert dgrad["items"] >= min_items, (dgrad, min_items)
    res = ternary((B, Cout, Ho, Wo), gen) if residual else None
    # a LeakyReLU backward hands multiples of bf16(0.2) = 205/1024 to the weight gradient: keep every channel's sum of
    # |dpre| below 2^14 so that its partial sums stay exact in fp32
    dy = ternary((B, Cout, Ho, Wo), gen, density=min(2.0 / 3.0, 8192.0 / (B * Ho * Wo)) if act == ACT_LRELU else 2.0 / 3.0)
    y_r, dx_r, dw_r, db_r, dpre = conv_reference(x.cuda(), w.cuda(), bias.cuda(), stride, pad, act, dy.cuda(),
                                                 res.cuda() if residual else None, relu_in)
    assert float(y_r.abs().max()) <= 256 and float(dx_r.abs().max()) <= 256
    q = 1024.0 if act == ACT_LRELU else 1.0
    assert float(dpre.abs().sum(dim=(0, 2, 3)).max()) * q < 2 ** 24 and B * Ho * Wo < 2 ** 24
    cin = max(Cin, cpad)
    xc = nhwc_dev(x, cin).requires_grad_()
    wc, bc = w.cuda().requires_grad_(), bias.cuda().requires_grad_()
    rc = nhwc_dev(res).requires_grad_() if residual else None
    cfg = ops.ConvCfg(k, k, stride, pad, act, relu_in, cpad)
    with ops.force_impl(L.IMPL_TC):
        y = ops.tap_conv(xc, cfg, (wc,), (bc,), None, rc)
        y.backward(nhwc_dev(dy))
    torch.cuda.synchronize()
    pairs = [(y, to_nhwc(y_r), "forward y", fwd),
             (xc.grad, to_nhwc(F.pad(dx_r, (0, 0, 0, 0, 0, cin - Cin))), "data gradient dx", dgrad if stride == 1 else None),
             (wc.grad, dw_r, "weight gradient dW", None), (bc.grad, db_r, "bias gradient db", None)]
    if residual:
        pairs.append((rc.grad, to_nhwc(dy), "residual gradient", None))
    assert_exact(pairs)


# (name, B, Cin, Cout, H, W, k, stride, pad, act, options).  Shapes of the benchmarked step's layers, sized so that each
# forward launch has >= 3 work items per SM whatever tile is picked; the comment names the forward instantiation
# tapconv_fwd_kernel<BN, ACT, MODE, HALO> the benchmark launches for that layer.
PERSISTENT_CASES = [
    ("256to256_3x3", 2, 256, 256, 160, 192, 3, 1, 1, ACT_NONE, {}),                      # <256,0,0,0>
    ("128to128_3x3_swapped", 2, 128, 128, 192, 320, 3, 1, 1, ACT_NONE, {}),             # <128,0,3,0>, mt = 2
    ("128to64_3x3_swapped", 2, 128, 64, 192, 320, 3, 1, 1, ACT_NONE, {}),               # <128,0,3,0>, mt = 2
    ("64to64_3x3_residual", 2, 64, 64, 192, 320, 3, 1, 1, ACT_NONE, {"residual": True}),  # <64,0,0,0> SIDE 2
    ("64to64_3x3_relu_mask_dgrad", 2, 64, 64, 192, 320, 3, 1, 1, ACT_NONE, {"relu_in": True}),  # dgrad <64,0,0,0> SIDE 1
    ("128to64_1x1_shortcut", 2, 128, 64, 192, 320, 1, 1, 0, ACT_NONE, {}),              # K = 128: stays on <64,0,0,0>
    ("128to256_3x3", 2, 128, 256, 160, 192, 3, 1, 1, ACT_NONE, {}),                     # <256,0,0,0>; gamma|beta of C = 128
    ("D0_5pad16to64_4x4s2_lrelu", 8, 5, 64, 320, 192, 4, 2, 2, ACT_LRELU, {"cpad": 16}),  # <64,1,0,0>, K = 4 x 64
    ("64to128_4x4s2_space_to_depth", 8, 64, 128, 320, 192, 4, 2, 2, ACT_NONE, {}),      # <128,0,3,0> on the s2d map
    ("128to128_odd_tiles_m", 1, 128, 128, 889, 128, 3, 1, 1, ACT_NONE, {}),             # 889 tiles: last work item half empty
    ("256to256_ragged_batch_tiles", 48, 256, 256, 37, 45, 3, 1, 1, ACT_NONE, {}),       # 9x2x7 tiles: ragged bottom and batch
]


def persistent_case_ids():
    return [c[0] for c in PERSISTENT_CASES]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PERSISTENT_CASES, ids=persistent_case_ids())
def test_tap_conv_exact_persistent(S, case):
    name, B, Cin, Cout, H, W, k, stride, pad, act, opt = case
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act, seed=zlib.crc32(name.encode()) % 1000, min_items=3 * sms, **opt)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TC_CASES)
def test_tap_conv_exact_small(S, case):
    B, Cin, Cout, H, W, k, stride, pad, act = case
    run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act, seed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MT_WGRAD_CASES)
def test_tap_conv_exact_multitap_wgrad(S, case):
    """Both weight-gradient kernels of narrow layers: several taps per CTA (default) and one tap per CTA (debug key 5 = 1)."""
    L, ops = S
    B, Cin, Cout, H, W, k, stride, pad, act = case
    run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act, seed=2)
    L.call("s2e_debug_set", 5, 1)
    try:
        run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act, seed=2)
    finally:
        L.call("s2e_debug_set", 5, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", HALO_CASES)
def test_tap_conv_exact_halo(S, case):
    L, ops = S
    B, Cin, Cout, H, W, k, stride, pad, act = case
    ops.set_halo(True)
    try:
        run_tap_case(S, B, Cin, Cout, H, W, k, stride, pad, act, seed=3, halo=True)
    finally:
        ops.set_halo(False)


# ------------------------------------------------------------------------------------------ mlp_shared (im2col GEMM)
@pytest.mark.gpu
def test_seg_im2col_gemm_exact_persistent(S):
    """SPADE's mlp_shared as the benchmark runs it: ReLU(conv3x3(one-hot segmap) + b) as a K = 64 GEMM on the segmap's
    im2col, the bias carried through the GEMM by the constant-one columns 62 / 63 (<128,2,3,0>), and the weight gradient
    of a ReLU-masked output gradient (the consumer applies the mask: act_grad_fused)."""
    L, ops = S
    gen = torch.Generator().manual_seed(5)
    B, C, hd, wd, Cout = 2, 4, 192, 320, 128
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    geom = fwd_launch(B, hd, wd, Cout, 64, 1, sms=sms)
    assert geom["items"] >= 3 * sms and work_items_lower_bound(B, hd, wd, Cout) >= 3 * sms, geom
    seg = F.one_hot(torch.randint(0, C, (B, 2 * hd, 2 * wd), generator=gen), C).permute(0, 3, 1, 2).float()
    bias = int_bias(Cout, gen)
    w = sparse_weight(Cout, C, 3, 3, gen, bias)
    segr = F.interpolate(seg, size=(hd, wd), mode="nearest").cuda()
    with exact_reference():
        v = F.conv2d(segr.double(), w.cuda().double(), bias.cuda().double(), padding=1)
    y_r = act_fwd_ref(v, ACT_RELU)
    dy = ternary((B, Cout, hd, wd), gen).cuda() * (y_r > 0)
    wr, br = w.cuda().double().requires_grad_(), bias.cuda().double().requires_grad_()
    with exact_reference():
        F.conv2d(segr.double(), wr, br, padding=1).backward(dy.double())
    col = ops.seg_im2col(seg.cuda(), hd, wd)
    wc, bc = w.cuda().requires_grad_(), bias.cuda().requires_grad_()
    with ops.force_impl(L.IMPL_TC):
        y = ops.SegConvFn.apply(col, wc, bc, L.ACT_RELU, True)
        y.backward(nhwc_dev(dy))
    torch.cuda.synchronize()
    assert_exact([(y, to_nhwc(y_r), "forward y", geom), (wc.grad, wr.grad, "weight gradient dW", None),
                  (bc.grad, br.grad, "bias gradient db", None)])


# ------------------------------------------------------------------------------------------ fused SPADE epilogues
# (C, B, H, W): gamma|beta = one N tile of 2C channels (<128,0,1|2,0> for C = 64, <256,0,1|2,0> for C = 128), tiles of one
# image row block; B = 2 so that every CTA's tiles span both samples and the per-sample constants change between tiles.
SPADE_SHAPES = {64: (2, 192, 320), 128: (2, 160, 192)}
SPADE_CASES = [(64, False, ACT_LRELU), (64, True, ACT_NONE), (128, False, ACT_NONE), (128, True, ACT_LRELU)]


def unpack_mask(amask, shape):
    """One bit per output element (bit e of byte j = channel 8j + e) -> bool NHWC."""
    bits = (amask.view(-1, 1).int() >> torch.arange(8, device=amask.device).view(1, 8)) & 1
    return bits.view(shape).bool()


def spade_modulation_check(S, out, gamma_r, beta_r, x_up, style, mean, rstd, act, what):
    """out (bf16, from the kernel) against float64 act(0.5 * [(x*ka + kb)(1 + gamma) + beta + s1 + x*kc]) evaluated from the
    exact gamma / beta and the kernel's own mean / rstd (ka = rstd, kb = -mean*rstd, kc = 1 + s0 as s2e_spade_params forms
    them in fp32).

    Bound: the epilogue forms the value with at most eight fp32 roundings (beta's bias + s1, the accumulator + that, the
    two FMAs, x*kc, the sum, 0.2f*o), each at most 2^-24 of a partial result, and every partial result is at most
    Sabs = 0.5*[(|x ka| + |kb|)|1 + gamma| + |beta| + |s1| + |x kc|] (0.2 |o| <= Sabs too): fp32 error <= e32 = 8 * 2^-24 * Sabs.
    The bf16 store then adds at most half a bf16 ulp of the fp32 value.  The test allows e32 + 2^-8 (|ref| + e32): one full
    bf16 ulp plus the fp32 term, which is 2^-16 of a bf16 ulp of Sabs."""
    L, ops = S
    B, H, W, C = out.shape
    par = torch.empty(B, 4, C, dtype=torch.float32, device="cuda")
    L.call("s2e_spade_params", L.ptr(mean), L.ptr(rstd), L.ptr(style), B, C, 0, L.ptr(par), L.stream())
    par = par.double()
    ka, kb, kc, s1 = [par[:, i].view(B, 1, 1, C) for i in range(4)]
    x = x_up.double()
    g1 = 1.0 + gamma_r.double()
    bt = beta_r.double() + s1
    o = 0.5 * ((x * ka + kb) * g1 + bt + x * kc)
    s_abs = 0.5 * ((x * ka).abs() + kb.abs()) * g1.abs() + 0.5 * (beta_r.double().abs() + s1.abs() + (x * kc).abs())
    if act == ACT_LRELU:
        o = torch.maximum(o, o * float(LRELU_SLOPE))
    e32 = 8 * U32 * s_abs
    tol = e32 + BF16_ULP_REL * (o.abs() + e32)
    err = (out.double() - o).abs()
    bad = err > tol
    n = int(bad.sum())
    if n:
        first = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError("%s: %d of %d elements outside the bound; first at %s: got %r, want %r +- %r" % (
            what, n, out.numel(), first, float(out[first]), float(o[first]), float(tol[first])))


def spade_inputs(C, up, seed):
    gen = torch.Generator().manual_seed(seed)
    B, H, W = SPADE_SHAPES[C]
    hx, wx = (H // 2, W // 2) if up else (H, W)
    Ca = 128
    actv = ternary((B, Ca, H, W), gen, nonneg=True)        # ReLU(mlp_shared(.)): {0, 1}
    bias = int_bias(2 * C, gen)
    w = sparse_weight(2 * C, Ca, 3, 3, gen, bias)          # gamma | beta weights packed along Cout (one budget per input channel)
    x = ternary((B, C, hx, wx), gen) + torch.randint(-1, 2, (1, C, 1, 1), generator=gen).float()   # integer-valued
    style = torch.randn(B, 2 * C, generator=gen) * 0.5
    dout = ternary((B, C, H, W), gen)
    return dict(B=B, H=H, W=W, actv=actv, w=w, bias=bias, x=x, style=style, dout=dout)


def gamma_beta_reference(inp, C):
    with exact_reference():
        gb = F.conv2d(inp["actv"].cuda().double(), inp["w"].cuda().double(), inp["bias"].cuda().double(), padding=1)
    return to_nhwc(gb[:, :C]), to_nhwc(gb[:, C:])


@pytest.mark.gpu
@pytest.mark.parametrize("C,up,act", SPADE_CASES)
def test_spade_conv_fused_exact_persistent(S, monkeypatch, C, up, act):
    """SpadeConvFn (training, MODE 2) and spade_conv_fused (no grad, MODE 1) across tiles and samples.  Exact: the gamma
    buffer (the integer gamma|beta convolution plus its bias), the activation bit mask against the sign of the kernel's
    own output.  Bounded per element: the modulated output (spade_modulation_check), and the gamma|beta convolution's data
    and weight gradients against float64 from the kernel's own dgamma|dbeta (see below).  The normalisation kernels
    (statistics, dx, dstyle) are covered elsewhere."""
    L, ops = S
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    inp = spade_inputs(C, up, seed=7 + C + int(up))
    B, H, W = inp["B"], inp["H"], inp["W"]
    tw, th = ops._fused_tile(H, W, C)
    geom = fwd_launch(B, H, W, 2 * C, 128, 9, spade=True, tile=(tw, th, 1), sms=sms)
    assert geom["items"] >= 3 * sms and work_items_lower_bound(B, H, W, 2 * C) >= 3 * sms, geom
    gamma_r, beta_r = gamma_beta_reference(inp, C)
    assert float(torch.cat([gamma_r, beta_r]).abs().max()) <= 256
    ccfg = ops.ConvCfg(3, 3, 1, 1, L.ACT_NONE, True)       # as the generator runs it: actv = ReLU(.), mask fused in dgrad
    cfg = ops.NormCfg(False, act, True, 0.1, 1e-5)
    xc = nhwc_dev(inp["x"])
    x_up = F.interpolate(inp["x"], scale_factor=2, mode="nearest") if up else inp["x"]
    x_up = to_nhwc(x_up).cuda()
    sc = inp["style"].cuda()
    wg, wb = inp["w"][:C].cuda(), inp["w"][C:].cuda()
    bg, bb = inp["bias"][:C].cuda(), inp["bias"][C:].cuda()

    # ---- no-grad fused kernel (MODE 1)
    with torch.no_grad():
        out1 = ops.spade_conv_fused(nhwc_dev(inp["actv"]), ccfg._replace(relu_in=False), (wg, wb), (bg, bb), xc, sc, cfg,
                                    None, None, None, up)
        mean1, rstd1, _ = ops.spade_statistics(xc, cfg, None, None, None, up)
    torch.cuda.synchronize()
    spade_modulation_check(S, out1, gamma_r, beta_r, x_up, sc, mean1, rstd1, act, "MODE 1 output")

    # ---- training kernel (MODE 2) and its backward
    seen = {}
    orig = ops._spade_style_bwd

    def capture(*args):
        orig(*args)
        seen["dgb"] = args[15].clone()           # dgamma | dbeta as the SPADE+Style backward hands it to the convolution

    monkeypatch.setattr(ops, "_spade_style_bwd", capture)
    ac = nhwc_dev(inp["actv"]).requires_grad_()
    wgc, wbc, bgc, bbc = [t.clone().requires_grad_() for t in (wg, wb, bg, bb)]
    out = ops.SpadeConvFn.apply(ac, xc, sc, wgc, wbc, bgc, bbc, ccfg, cfg, None, None, None, up, None)
    _, _, gamma, _, mean, rstd, amask = out.grad_fn.saved_tensors
    torch.cuda.synchronize()
    assert_exact([(gamma, gamma_r, "MODE 2 gamma buffer", geom)])
    spade_modulation_check(S, out, gamma_r, beta_r, x_up, sc, mean, rstd, act, "MODE 2 output")
    if act != ACT_NONE:
        assert_exact([(unpack_mask(amask, out.shape).float(), (out.float() > 0).float(), "MODE 2 activation mask", geom)])
    out.backward(nhwc_dev(inp["dout"]))
    torch.cuda.synchronize()
    dgb = seen["dgb"].float().permute(0, 3, 1, 2).double()     # NCHW, bf16 values
    conv_grad_check(ac.grad, wgc.grad, wbc.grad, inp, dgb, C)


def conv_grad_check(dactv, dwg, dwb, inp, dgb, C):
    """Data gradient (ReLU-masked by actv > 0) and weight gradient of the gamma|beta convolution for a bf16 dgamma|dbeta that
    is not integer-valued, per element against float64.  Bound: a sum of n non-zero products accumulated in fp32 in any
    order is off by at most n * 2^-24 * sum |products| (n counted per element from the non-zero patterns); the data
    gradient's bf16 store adds at most one bf16 ulp.  The integer-valued tap-convolution cases run the same kernels at
    these shapes exactly."""
    actv = inp["actv"].cuda().double()
    w = inp["w"].cuda().double()
    with exact_reference():
        dx = torch.nn.grad.conv2d_input(actv.shape, w, dgb, padding=1) * (actv > 0)
        dx_abs = torch.nn.grad.conv2d_input(actv.shape, w.abs(), dgb.abs(), padding=1)
        dx_n = torch.nn.grad.conv2d_input(actv.shape, w.ne(0).double(), dgb.ne(0).double(), padding=1)
        dw = torch.nn.grad.conv2d_weight(actv, w.shape, dgb, padding=1)
        dw_abs = torch.nn.grad.conv2d_weight(actv, w.shape, dgb.abs(), padding=1)         # actv >= 0
        dw_n = torch.nn.grad.conv2d_weight(actv.ne(0).double(), w.shape, dgb.ne(0).double(), padding=1)
    e_dx = dx_n * U32 * dx_abs
    checks = [(dactv.double().permute(0, 3, 1, 2), dx,
               e_dx + BF16_ULP_REL * (dx.abs() + e_dx), "data gradient d actv"),
              (torch.cat([dwg, dwb]).double(), dw, dw_n * U32 * dw_abs, "weight gradient d W_gamma|beta")]
    errs = []
    for got, ref, tol, what in checks:
        bad = (got - ref).abs() > tol
        n = int(bad.sum())
        if n:
            first = tuple(int(i) for i in bad.nonzero()[0])
            errs.append("%s: %d elements outside the bound; first at %s: got %r, want %r +- %r" % (
                what, n, first, float(got[first]), float(ref[first]), float(tol[first])))
    assert not errs, "\n".join(errs)


# ------------------------------------------------------------------------------------------ CPU-side checks of the oracle
def test_builder_respects_its_bounds():
    gen = torch.Generator().manual_seed(0)
    for (Cout, Cin, k, extra) in [(256, 256, 3, 0), (64, 64, 3, 1), (128, 4, 3, 0), (64, 16, 4, 0), (512, 128, 3, 0)]:
        bias = int_bias(Cout, gen)
        w = sparse_weight(Cout, Cin, k, k, gen, bias, extra=extra)
        row, col = check_weight_bounds(w, bias, extra)
        assert 0 < row and 0 < col <= 256
        # the largest |result| the weights allow: all-ones input / output gradient, every product counted positively
        y_max = F.conv2d(torch.ones(1, Cin, 2 * k, 2 * k).double(), w.abs().double(), bias.abs().double())
        assert float(y_max.max()) + extra <= 256
        dx_max = torch.nn.grad.conv2d_input((1, Cin, 3 * k, 3 * k), w.abs().double(), torch.ones(1, Cout, 2 * k + 1, 2 * k + 1).double())
        assert float(dx_max.max()) <= 256
    # a dense request is cut down to the budgets
    w = sparse_weight(64, 256, 3, 3, gen, torch.full((64,), 3.0), target=10 ** 6)
    row, col = check_weight_bounds(w, torch.full((64,), 3.0))
    assert row == 253 and col <= 256
    with pytest.raises(AssertionError):
        check_weight_bounds(torch.ones(8, 64, 3, 3))
    with pytest.raises(AssertionError):
        check_weight_bounds(torch.ones(300, 1, 1, 1))
    w = sparse_weight(512, 16, 3, 3, gen, target=10 ** 6)     # the input-channel budget binds (9 x 512 taps per channel)
    assert check_weight_bounds(w)[1] == 256
    # the exact reference results of a small case are integers within +-256 (weight gradient: within the pixel count)
    B, H, W = 2, 9, 7
    x = ternary((B, 64, H, W), gen)
    bias = int_bias(64, gen)
    w = sparse_weight(64, 64, 3, 3, gen, bias)
    y, dx, dw, db, _ = conv_reference(x, w, bias, 1, 1, ACT_NONE, ternary((B, 64, H, W), gen))
    for t, lim in ((y, 256), (dx, 256), (dw, B * H * W), (db, B * H * W)):
        assert torch.equal(t.double(), t.double().round()) and float(t.abs().max()) <= lim
    assert float(y.abs().max()) > 0 and float(dw.abs().max()) > 0


def test_comparator_flags_single_and_block_errors():
    gen = torch.Generator().manual_seed(1)
    B, Cin, Cout, H, W = 2, 128, 64, 12, 20
    x = ternary((B, Cin, H, W), gen)
    bias = int_bias(Cout, gen)
    w = sparse_weight(Cout, Cin, 3, 3, gen, bias)
    y = to_nhwc(F.conv2d(x.double(), w.double(), bias.double(), padding=1)).float()
    geom = fwd_launch(B, H, W, Cout, Cin, 9)
    assert mismatch(y.clone(), y, "y", geom) is None
    off = y.clone()
    off[1, 7, 13, 40] += 1
    msg = mismatch(off, y, "y", geom)
    assert msg is not None and "1 of" in msg and "(1, 7, 13, 40)" in msg and "pixel tile" in msg
    # one 64-channel block of one tap dropped for one pixel tile
    w_drop = w.clone()
    w_drop[:, 64:128, 0, 2] = 0
    y_drop = to_nhwc(F.conv2d(x.double(), w_drop.double(), bias.double(), padding=1)).float()
    tw, th, tb = geom["tw"], geom["th"], geom["tb"]
    bad = y.clone()
    bad[:tb, :th, :tw] = y_drop[:tb, :th, :tw]
    msg = mismatch(bad, y, "y", geom)
    assert msg is not None and "pixel tile 0 " in msg, msg
    with pytest.raises(AssertionError):
        assert_exact([(bad, y, "y", geom)])
    assert_exact([(y, y.clone(), "y", geom)])


def test_persistent_cases_meet_work_item_bound_on_b200():
    """Each persistent-regime shape gives >= 3 work items per SM on a 148-SM B200, whatever tile is picked."""
    need = 3 * B200_SMS
    for name, B, Cin, Cout, H, W, k, stride, pad, act, opt in PERSISTENT_CASES:
        fwd, dgrad, (Ho, Wo) = tap_geometries(B, Cin, Cout, H, W, k, stride, pad, opt.get("cpad", 0), opt.get("residual", False),
                                              opt.get("relu_in", False))
        assert work_items_lower_bound(B, Ho, Wo, Cout) >= need, name
        assert fwd["items"] >= work_items_lower_bound(B, Ho, Wo, Cout) and fwd["items"] >= need, (name, fwd)
    for C, (B, H, W) in SPADE_SHAPES.items():
        tw = min(W, 128)
        while W % tw or 128 % tw:
            tw -= 1
        geom = fwd_launch(B, H, W, 2 * C, 128, 9, spade=True, tile=(tw, 128 // tw, 1))
        assert geom["items"] >= need and work_items_lower_bound(B, H, W, 2 * C) >= need, (C, geom)
        assert (geom["tiles_w"] * geom["tiles_h"]) % geom["mt"] == 0            # the kernel's requirement
    assert fwd_launch(2, 192, 320, 128, 64, 1)["items"] >= need                # mlp_shared
    # the geometry each special case is there for
    g = {c[0]: tap_geometries(*c[1:9], opt.get("cpad", 0), opt.get("residual", False), opt.get("relu_in", False))
         for c in PERSISTENT_CASES for opt in [c[10]]}
    odd = g["128to128_odd_tiles_m"][0]
    assert odd["tiles_m"] % 2 == 1 and odd["mt"] == 2 and odd["bn"] == 128
    rag = g["256to256_ragged_batch_tiles"][0]
    assert rag["tb"] > 1 and 48 % rag["tb"] and 37 % rag["th"] and rag["mt"] == 1
    assert g["64to64_3x3_residual"][0]["bn"] == 64 and g["64to64_3x3_relu_mask_dgrad"][1]["bn"] == 64
    assert g["128to64_1x1_shortcut"][0]["bn"] == 64
    assert g["D0_5pad16to64_4x4s2_lrelu"][0]["bn"] == 64
    assert g["128to128_3x3_swapped"][0]["mt"] == 2 and g["256to256_3x3"][0]["bn"] == 256


@pytest.fixture(scope="module")
def S():
    from seg2eye_b200 import _lib as L, ops
    L.lib()
    return L, ops
