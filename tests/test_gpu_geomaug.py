"""`--diff_augment xflip,geometric` on the device: the draw against `s2e_diffaug_draw_p` and a NumPy restatement (gates
and coin bit for bit, M within 2 fp32 ulp of an fp64 composition, gate frequencies, normals); the layout kernel against
today's masked kernel, the exact index mirror and a float64 restatement (forced near-90/180 degree rotations and the
extreme zoom-out included); the deterministic adjoint against a float64 scatter restatement and the adjoint identity;
one G and one D step against the model fed the restatement; the C-ABI call trace; CUDA-graph replays; ADA under graphs;
and two ranks against one process."""
import contextlib
import datetime
import io
import math
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import seg2eye_oracle as O
from test_gpu_diffaug import (COLOR, CUTOUT, NAMES, TRANSLATION, _bf16_ulp, _free_port, _inputs, _load, _means, _opts,
                              _philox4x32_10, _rel, _sds, _state, _traced_step, _trainer, _unit)

pytestmark = pytest.mark.gpu

XFLIP, GEOMETRIC = 8, 16
ALL = COLOR | XFLIP | GEOMETRIC | TRANSLATION | CUTOUT


def _p(v):
    return torch.tensor([v], dtype=torch.float64, device="cuda")


# ------------------------------------------------------------------------------------------ NumPy restatement of the draw
def _sinpi(t):
    return np.where(np.mod(t, 1.0) == 0, 0.0, np.sin(np.pi * t))


def _cospi(t):
    return np.where(np.mod(t + 0.5, 1.0) == 0, 0.0, np.cos(np.pi * t))


def _box_muller(ra, rb):
    u = ((ra >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24
    v = ((rb >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24
    rad = np.sqrt(-2.0 * np.log(u))
    return rad * _cospi(2.0 * v), rad * _sinpi(2.0 * v)


def np_geom(seed, counter, offset, B, H, W, p):
    """-> M [B, 6] (fp64 composition), the XFLIP / GEOMETRIC bits, the seven gates and the four normals, per the header."""
    s, c = seed % 2 ** 64, counter % 2 ** 64
    key = (s & 0xFFFFFFFF, s >> 32)
    idx = np.arange(offset, offset + B, dtype=np.uint64)
    lo, hi = np.full(B, c & 0xFFFFFFFF, np.uint64), np.full(B, c >> 32, np.uint64)
    r2, r3, r4, r5 = (_philox4x32_10([idx, lo, hi, np.full(B, k, np.uint64)], key) for k in (2, 3, 4, 5))
    u = lambda r: _unit(r).astype(np.float64)     # noqa: E731
    p_rot = 1.0 - math.sqrt(max(1.0 - p, 0.0))
    gates = dict(xflip=u(r2[1]) < p, coin=u(r2[2]) < 0.5, scale=u(r2[3]) < p, rot1=u(r3[0]) < p_rot, aniso=u(r3[1]) < p,
                 rot2=u(r3[2]) < p_rot, xfrac=u(r3[3]) < p)
    n0, n1 = _box_muller(r4[0], r4[1])
    n2, n3 = _box_muller(r5[0], r5[1])
    mirror = gates["xflip"] & gates["coin"]
    is_ = np.where(gates["scale"], np.exp2(-0.2 * n0), 1.0)
    ia = np.where(gates["aniso"], np.exp2(-0.2 * n1), 1.0)
    t1 = np.where(gates["rot1"], 2.0 * u(r4[2]) - 1.0, 0.0)
    t2 = np.where(gates["rot2"], 2.0 * u(r4[3]) - 1.0, 0.0)
    s1, c1, s2, c2 = _sinpi(t1), _cospi(t1), _sinpi(t2), _cospi(t2)
    b00, b01, b10, b11 = c1 * ia, s1 / ia, -s1 * ia, c1 / ia
    f = np.where(mirror, -is_, is_)
    a00, a01 = f * (b00 * c2 - b01 * s2), f * (b00 * s2 + b01 * c2)
    a10, a11 = is_ * (b10 * c2 - b11 * s2), is_ * (b10 * s2 + b11 * c2)
    dx = np.where(gates["xfrac"], -0.125 * n2 * W, 0.0)
    dy = np.where(gates["xfrac"], -0.125 * n3 * H, 0.0)
    M = np.stack([a00, a01, a00 * dx + a01 * dy, a10, a11, a10 * dx + a11 * dy], 1)
    geo = gates["scale"] | gates["rot1"] | gates["aniso"] | gates["rot2"] | gates["xfrac"]
    bits = (mirror * XFLIP | geo * GEOMETRIC).astype(np.int32)
    return M, bits, gates, (n0, n1, n2, n3)


def test_draw_keeps_todays_records_and_gates_and_matches_numpy():
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    for H, W in ((640, 384), (41, 33)):
        for seed in (0, -1, 0x0123456789ABCDEF):
            for counter in (0, 77777, 2 ** 32 + 7):
                for offset, B in ((0, 16), (2 ** 31 + 9, 37), (2 ** 32 - 4, 4)):
                    for p in (0.0, 0.3, 1.0):
                        st_a, st_b = _state(seed, counter), _state(seed, counter)
                        rec_a, mask_a = ops.diffaug_draw_p(st_a, _p(p), B, offset, H, W)
                        rec_b, geom, mask_b = ops.diffaug_draw_geom(st_b, _p(p), B, offset, H, W)
                        assert rec_b.cpu().numpy().tobytes() == rec_a.cpu().numpy().tobytes()
                        assert st_a.tolist() == st_b.tolist() == [seed, counter + 1]
                        mb = mask_b.cpu().numpy()
                        assert np.array_equal(mb & 7, mask_a.cpu().numpy())
                        M, bits, _, _ = np_geom(seed, counter, offset, B, H, W, p)
                        assert np.array_equal(mb & 24, bits), (seed, counter, offset, p)
                        g = geom.cpu().numpy()
                        assert (g[:, 6:] == 0).all()
                        ulp = np.spacing(np.abs(M).astype(np.float32)).astype(np.float64)
                        err = np.abs(g[:, :6].astype(np.float64) - M)
                        assert (err <= 2 * ulp).all(), (seed, counter, offset, p, float((err / ulp).max()))
                        if p == 0.0:
                            assert not bits.any() and (g[:, :6] == [1, 0, 0, 0, 1, 0]).all()
                        if p == 1.0:
                            assert (bits & GEOMETRIC).all()


def test_gate_frequencies_and_normals():
    from scipy import stats
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    H, W, n = 384, 640, 1 << 15
    for p in (0.3, 1.0):
        st = _state(20201207, 11)
        draws = [ops.diffaug_draw_geom(st, _p(p), 4096, 0, H, W) for _ in range(n // 4096)]
        masks = torch.cat([d[2] for d in draws]).cpu().numpy()
        geom = torch.cat([d[1] for d in draws]).double().cpu().numpy()
        gates = {}
        for k in range(n // 4096):       # the restated gates, whose combination the device reproduces bit for bit
            _, bits, g, _ = np_geom(20201207, 11 + k, 0, 4096, H, W, p)
            assert np.array_equal(masks[4096 * k:4096 * (k + 1)] & 24, bits)
            for name, v in g.items():
                gates.setdefault(name, []).append(v)
        p_rot = 1 - math.sqrt(1 - p)
        for name, q in dict(xflip=p, coin=0.5, scale=p, rot1=p_rot, aniso=p, rot2=p_rot, xfrac=p).items():
            cnt = int(np.concatenate(gates[name]).sum())
            assert abs(cnt - n * q) <= 5 * (n * q * (1 - q)) ** 0.5 + 1e-9, (p, name, cnt)
        for bit, q in ((XFLIP, p / 2), (GEOMETRIC, 1 - (1 - p) ** 4)):
            cnt = int(((masks & bit) != 0).sum())
            assert abs(cnt - n * q) <= 5 * (n * q * (1 - q)) ** 0.5 + 1e-9, (p, bit, cnt)
        if p == 1.0:     # every gate on: the normals from the device's M (det = +-1/s^2, t = A d, d = -0.125 n (W, H))
            A = geom[:, [0, 1, 3, 4]].reshape(-1, 2, 2)
            det = np.linalg.det(A)
            d = np.linalg.solve(A, geom[:, [2, 5]][..., None])[..., 0]
            n0 = -2.5 * np.log2(np.abs(det))
            n2, n3 = -8.0 * d[:, 0] / W, -8.0 * d[:, 1] / H
            sv = np.linalg.svd(A, compute_uv=False)
            absn1 = 2.5 * np.log2(sv[:, 0] / sv[:, 1])            # |n1|: the anisotropy's sign is not recoverable
            for v in (n0, n2, n3):
                assert stats.kstest(v, "norm").pvalue > 1e-4
            assert stats.kstest(absn1, stats.halfnorm.cdf).pvalue > 1e-4
            assert np.abs(np.concatenate([n0, n2, n3])).max() <= 5.95


# ------------------------------------------------------------------------------------------ float64 restatement
def _fold(k, n):
    m = 2 * (n - 1)
    q = torch.remainder(k, m)
    return torch.where(q < n, q, m - q)


def _warp(m, si, sj, H, W):
    """The kernel's fp32 coordinates, one rounding per operation (separate torch kernels do not contract)."""
    hx = torch.tensor(0.5 * (W - 1), dtype=torch.float32, device=m.device)
    hy = torch.tensor(0.5 * (H - 1), dtype=torch.float32, device=m.device)
    xc, yc = sj.float() - hx, si.float() - hy
    X = ((m[0] * xc + m[1] * yc) + m[2]) + hx
    Y = ((m[3] * xc + m[4] * yc) + m[5]) + hy
    return X, Y


def _matrix(geom, mask, b, policy):
    m = geom[b, :6].float().clone()
    if int(mask[b]) & XFLIP and not policy & XFLIP:
        m[:3] = -m[:3]
    return m


def ref_geom(seg, fake, real, rec, geom, mask, policy, cpad, means=None):
    """The augmented D input in float64 torch (differentiable in fake), NHWC with cpad channels, from the kernel's fp32
    coordinates: labels at the folded nearest tap, the image bilinear in float64 at the folded taps, then colour."""
    B, nc, H, W = seg.shape
    dev = seg.device
    ii = torch.arange(H, device=dev)[:, None].expand(H, W)
    jj = torch.arange(W, device=dev)[None, :].expand(H, W)
    rows = []
    for row in range(2 * B):
        b = row % B
        pb = policy & int(mask[b])
        x = (fake if row < B else real)[b, 0].double()
        lab = seg[b].double()
        r = rec[b].double()
        si, sj, keep = ii, jj, torch.ones(H, W, dtype=torch.bool, device=dev)
        if pb & TRANSLATION:
            si, sj = ii + int(rec[b, 2]), jj + int(rec[b, 3])
            keep = keep & (si >= 0) & (si < H) & (sj >= 0) & (sj < W)
        if pb & CUTOUT:
            cx, cy = int(H / 2 + 0.5), int(W / 2 + 0.5)
            x0, y0 = int(rec[b, 4]) - cx // 2, int(rec[b, 5]) - cy // 2
            keep = keep & ~((ii >= x0) & (ii < x0 + cx) & (jj >= y0) & (jj < y0 + cy))
        si, sj = si.clamp(0, H - 1), sj.clamp(0, W - 1)
        if pb & GEOMETRIC:
            X, Y = _warp(_matrix(geom, mask, b, policy), si, sj, H, W)
            li, lj = _fold(torch.floor(Y + 0.5).long(), H), _fold(torch.floor(X + 0.5).long(), W)
            x0f, y0f = torch.floor(X), torch.floor(Y)
            fx, fy = (X - x0f).double(), (Y - y0f).double()
            c0, c1 = _fold(x0f.long(), W), _fold(x0f.long() + 1, W)
            r0, r1 = _fold(y0f.long(), H), _fold(y0f.long() + 1, H)
            v = (1 - fy) * ((1 - fx) * x[r0, c0] + fx * x[r0, c1]) + fy * ((1 - fx) * x[r1, c0] + fx * x[r1, c1])
            labs = lab[:, li, lj]
        else:
            sjj = W - 1 - sj if pb & XFLIP else sj
            v, labs = x[si, sjj], lab[:, si, sjj]
        if pb & COLOR:
            mu = x.mean() if means is None else means[row].double()
            br, ct = r[0] - 0.5, r[1] + 0.5
            v = (v + br - (mu + br)) * ct + (mu + br)
        out = torch.cat([labs, v[None]]) * keep
        rows.append(out.permute(1, 2, 0))
    return torch.nn.functional.pad(torch.stack(rows), (0, cpad - (nc + 1)))


def _fwd(seg, fake, real, cpad, rec, mask, geom, policy):
    from seg2eye_b200 import ops
    return ops.MakeDInputAugGeomFn.apply(seg, fake, real, cpad, rec, mask, geom, policy)


def _check_forward(out, ref, fake, real, rec, policy, mask, nc):
    B = fake.shape[0]
    assert torch.equal(out[..., :nc], ref[..., :nc].to(torch.bfloat16))           # labels exactly
    assert torch.all(out[..., nc + 1:] == 0)
    for row in range(2 * B):
        b = row % B
        pb = policy & int(mask[b])
        got, want = out[row, ..., nc].double(), ref[row, ..., nc]
        if not pb & (GEOMETRIC | COLOR):
            assert torch.equal(got, want.to(torch.bfloat16).double()), row
            continue
        # one bf16 ulp, plus the kernel's fp32 interpolation and colour: 2^-18 (1 + c) max |image|
        c = float(rec[b, 1]) + 0.5 if pb & COLOR else 1.0
        amax = float((fake if row < B else real)[b].abs().max())
        bound = torch.maximum(_bf16_ulp(want), _bf16_ulp(got)) + 2.0 ** -18 * (1 + abs(c)) * amax
        d = (got - want).abs()
        assert torch.all(d <= bound), (row, float((d / bound).max()))


CASES = [(3, 4, 41, 33), (2, 4, 320, 256), (2, 4, 384, 640), (2, 35, 41, 33)]
POLICIES = [XFLIP, GEOMETRIC, XFLIP | GEOMETRIC, ALL, GEOMETRIC | TRANSLATION | CUTOUT, COLOR | GEOMETRIC]


@pytest.mark.parametrize("case", CASES)
def test_forward_without_new_bits_is_todays_masked_kernel_and_xflip_is_the_index_mirror(case):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    seg, fake, real = _inputs(B, nc, H, W, 5 + nc + H)
    cpad = -(-(nc + 1) // 16) * 16
    rec, geom, _ = ops.diffaug_draw_geom(_state(3 + H, 7), _p(1.0), B, 0, H, W)
    mask7 = torch.arange(B, dtype=torch.int32, device="cuda") % 8
    for policy in (ALL, COLOR | TRANSLATION | CUTOUT, TRANSLATION):
        a = ops.MakeDInputAugMaskedFn.apply(seg, fake, real, cpad, rec, mask7, policy & 7)
        assert torch.equal(_fwd(seg, fake, real, cpad, rec, mask7, geom, policy), a), policy
    # xflip alone: exactly the mirrored layout for mirrored samples, today's layout for the others
    mflip = torch.tensor([XFLIP * (b % 2) for b in range(B)], dtype=torch.int32, device="cuda")
    out = _fwd(seg, fake, real, cpad, rec, mflip, geom, XFLIP)
    plain = ops.MakeDInputFn.apply(seg, fake, real, cpad)
    flipped = ops.MakeDInputFn.apply(seg.flip(-1), fake.flip(-1), real.flip(-1), cpad)
    for row in range(2 * B):
        assert torch.equal(out[row], (flipped if row % B % 2 else plain)[row]), row
    # the mirror through the warp (M = F exactly) is the same bits
    eye_f = torch.tensor([-1, 0, 0, 0, 1, 0, 0, 0], dtype=torch.float32, device="cuda").repeat(B, 1)
    mboth = torch.full((B,), XFLIP | GEOMETRIC, dtype=torch.int32, device="cuda")
    assert torch.equal(_fwd(seg, fake, real, cpad, rec, mboth, eye_f, XFLIP | GEOMETRIC), flipped)


def _forced(kind, B, H, W):
    """Matrices forced to the hard cases: near-90 / near-180 degree rotations and the extreme zoom-out (s and a at their
    bounds 2^(0.2 * -5.9), rotated), with fractional translations."""
    z = 2.0 ** (0.2 * 5.9)
    out = []
    for b in range(B):
        if kind == "rot90":
            th, sc = math.pi / 2 - 1e-3 * (b + 1), (1.0, 1.0)
        elif kind == "rot180":
            th, sc = math.pi - 7e-4 * (b + 1), (1.0, 1.0)
        else:
            th, sc = 0.3 * b, (z * z, 1.0) if b % 2 else (z, z)
        c, s = math.cos(th), math.sin(th)
        A = np.array([[c, s], [-s, c]]) @ np.diag(sc)
        t = A @ np.array([0.37 * W / 8, -0.21 * H / 8])
        out.append([A[0, 0], A[0, 1], t[0], A[1, 0], A[1, 1], t[1], 0, 0])
    return torch.tensor(out, dtype=torch.float32, device="cuda")


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("source", ["drawn", "rot90", "rot180", "zoomout"])
def test_forward_matches_float64_restatement(case, source):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    seg, fake, real = _inputs(B, nc, H, W, 13 + nc + W)
    cpad = -(-(nc + 1) // 16) * 16
    st = _state(99 + H, 2 ** 32 + 5)
    for it in range(2):
        rec, geom, mask = ops.diffaug_draw_geom(st, _p(0.7), B, 0, H, W)
        if source != "drawn":
            geom = _forced(source, B, H, W)
            mask = mask | GEOMETRIC
        means = _means(fake, real)
        for policy in POLICIES:
            out = _fwd(seg, fake, real, cpad, rec, mask, geom, policy)
            ref = ref_geom(seg, fake, real, rec, geom, mask, policy, cpad, means)
            _check_forward(out, ref, fake, real, rec, policy, mask, nc)
        same = _fwd(seg, real, real, cpad, rec, mask, geom, ALL)      # rows b and B + b share M
        assert torch.equal(same[:B], same[B:])


# ------------------------------------------------------------------------------------------ adjoint
def _grad(seg, fake, real, cpad, rec, mask, geom, policy, g):
    f = fake.clone().requires_grad_(True)
    _fwd(seg, f, real, cpad, rec, mask, geom, policy).backward(g)
    return f.grad


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("source", ["drawn", "rot90", "rot180", "zoomout"])
def test_adjoint_matches_float64_scatter_and_the_identity(case, source):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    seg, fake, real = _inputs(B, nc, H, W, 29 + nc + H)
    cpad = -(-(nc + 1) // 16) * 16
    rec, geom, mask = ops.diffaug_draw_geom(_state(7 + W, 12), _p(0.8), B, 0, H, W)
    if source != "drawn":
        geom, mask = _forced(source, B, H, W), mask | GEOMETRIC
    gen = torch.Generator().manual_seed(H + W)
    g = torch.randn(2 * B, H, W, cpad, generator=gen).to(torch.bfloat16).cuda()
    x = torch.randn(B, 1, H, W, generator=gen, dtype=torch.float64).cuda()
    for policy in POLICIES:
        got = _grad(seg, fake, real, cpad, rec, mask, geom, policy, g).double()
        f64 = fake.double().requires_grad_(True)
        (ref_geom(seg, f64, real, rec, geom, mask, policy, cpad) * g.double()).sum().backward()
        want = f64.grad          # autograd's float64 scatter of w h into the folded taps
        f0 = torch.zeros_like(f64).requires_grad_(True)
        (ref_geom(seg, f0, real, rec, geom, mask, policy & ~COLOR, cpad) * g.double().abs()).sum().backward()
        wabs = f0.grad            # Warp^T |h|: the scale of the fp32 gather's rounding
        f1 = torch.zeros_like(f64).requires_grad_(True)
        (ref_geom(seg, f1, real, rec, geom, mask, policy & ~COLOR, cpad) * g.double()).sum().backward()
        mean = f1.grad.mean(dim=(1, 2, 3), keepdim=True).abs()      # sum(h) / HW: the weights sum to 1
        c = torch.tensor([float(rec[b, 1]) + 0.5 if policy & int(mask[b]) & COLOR else 1.0 for b in range(B)],
                         dtype=torch.float64, device="cuda").view(B, 1, 1, 1)
        bound = 2.0 ** -17 * (c.abs() * wabs + ((1 - c).abs() + 1) * mean) + 1e-30
        assert torch.all((got - want).abs() <= bound), (policy, float(((got - want).abs() / bound).max()))
        # <Aug x, g> = <x, Aug^T g> over the fake half, Aug the linear part of fake -> output
        zero = torch.zeros_like(real)
        tx = ref_geom(seg, x, zero, rec, geom, mask, policy, cpad) - ref_geom(seg, torch.zeros_like(x), zero, rec, geom, mask,
                                                                          policy, cpad)
        lhs = float((tx[:B, ..., nc] * g[:B, ..., nc].double()).sum())
        rhs = float((x * got).sum())
        assert abs(lhs - rhs) <= 1e-6 * float((x.abs() * got.abs()).sum()), (policy, lhs, rhs)


@pytest.mark.parametrize("hw", [(41, 33), (2, 2), (5, 3)])
def test_adjoint_counts_edge_rows_and_columns_once(hw):
    """Integer gradients and dyadic weights: every sum is exact, so the gather must equal the float64 scatter bit for bit.
    The identity warp (M = I, weight-1 taps on the edge rows and columns) returns g itself; the half-pixel shifts fold
    taps -1 and n onto rows / columns 1 and n-2 and leave the edges with one tap each."""
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    H, W = hw
    B, nc = 4, 4
    seg, fake, real = _inputs(B, nc, H, W, 3)
    cpad = 16
    rec = ops.diffaug_draw(_state(1, 1), B, 0, H, W)
    g = torch.randint(-4, 5, (2 * B, H, W, cpad), generator=torch.Generator().manual_seed(H)).to(torch.bfloat16).cuda()
    mask = torch.full((B,), GEOMETRIC, dtype=torch.int32, device="cuda")
    eye = torch.tensor([1, 0, 0, 0, 1, 0, 0, 0], dtype=torch.float32, device="cuda").repeat(B, 1)
    got = _grad(seg, fake, real, cpad, rec, mask, eye, GEOMETRIC, g)
    assert torch.equal(got[:, 0], g[:B, ..., nc].float())
    shifts = torch.tensor([[1, 0, -0.5, 0, 1, 0.5, 0, 0], [-1, 0, 0.5, 0, 1, -0.5, 0, 0], [1, 0, 0.25, 0, -1, -0.75, 0, 0],
                           [0.5, 0, 0, 0, 0.5, 0, 0, 0]], dtype=torch.float32, device="cuda")
    got = _grad(seg, fake, real, cpad, rec, mask, shifts, GEOMETRIC, g)
    f64 = fake.double().requires_grad_(True)
    (ref_geom(seg, f64, real, rec, shifts, mask, GEOMETRIC, cpad) * g.double()).sum().backward()
    assert torch.equal(got.double(), f64.grad)


def test_adjoint_is_deterministic_eager_and_replayed():
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = 4, 4, 320, 256
    seg, fake, real = _inputs(B, nc, H, W, 8)
    cpad = 16
    rec, geom, mask = ops.diffaug_draw_geom(_state(11, 3), _p(1.0), B, 0, H, W)
    g = torch.randn(2 * B, H, W, cpad, generator=torch.Generator().manual_seed(1)).to(torch.bfloat16).cuda()
    policy = ALL
    a = _grad(seg, fake, real, cpad, rec, mask, geom, policy, g)
    b = _grad(seg, fake, real, cpad, rec, mask, geom, policy, g)
    assert torch.equal(a, b)
    from seg2eye_b200 import _lib as L
    dfake = torch.empty(B, 1, H, W, device="cuda")
    scratch = torch.empty(B, dtype=torch.float64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):        # warm-up outside the capture
        L.call("s2e_d_input_grad_aug_geom", L.ptr(g), B, nc, H, W, cpad, L.ptr(rec), policy, L.ptr(mask), L.ptr(geom),
               L.ptr(scratch), L.ptr(dfake), L.stream())
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        L.call("s2e_d_input_grad_aug_geom", L.ptr(g), B, nc, H, W, cpad, L.ptr(rec), policy, L.ptr(mask), L.ptr(geom),
               L.ptr(scratch), L.ptr(dfake), L.stream())
    for _ in range(2):
        dfake.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(dfake, a)


# ------------------------------------------------------------------------------------------ model
FULL = "color,xflip,geometric,translation,cutout"


class _RestatedGeom:
    """Stands in for ops.MakeDInputAugGeomFn: the float64 restatement, rounded to bf16, with torch autograd to the fake."""

    @staticmethod
    def apply(seg, fake, real, cpad, params, opmask, geom, policy):
        return ref_geom(seg, fake, real, params, geom, opmask, policy, max(cpad, seg.shape[1] + 1)).to(torch.bfloat16).contiguous()


def test_model_steps_match_the_restated_d_input(tmp_path, monkeypatch):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    torch.cuda.set_device(0)
    oopt, opt = _opts(str(tmp_path), FULL)
    sds = _sds(oopt, 51)
    batch = O.synth_batch(oopt, 3, 54)
    res = {}
    for name in ("kernel", "restated"):
        with contextlib.redirect_stdout(io.StringIO()):
            m = Pix2PixModel(opt)
        _load(m, sds)
        m.diffaug_state.copy_(_state(2025, 3))
        m.train()
        with monkeypatch.context() as mp_:
            if name == "restated":
                mp_.setattr(ops, "MakeDInputAugGeomFn", _RestatedGeom)
            losses, fake = m({k: v.clone() for k, v in batch.items()}, mode="generator")
            fake.retain_grad()
            sum(losses.values()).mean().backward()
            d_losses = m({k: v.clone() for k, v in batch.items()}, mode="discriminator")
        torch.cuda.synchronize()
        res[name] = ({k: v.detach().reshape(-1)[0] for k, v in {**losses, **d_losses}.items()}, fake.grad.detach().clone(),
                     m.diffaug_state.tolist())
    (lk, gk, sk), (lr_, gr, sr) = res["kernel"], res["restated"]
    assert sk == sr == [2025, 5]
    print("losses kernel %s restated %s, dfake rel %.2e" % ({k: float(v) for k, v in lk.items()},
                                                           {k: float(v) for k, v in lr_.items()}, _rel(gk, gr)))
    for k in lk:    # the tolerances of tests/test_gpu_diffaug.py's model test
        assert abs(float(lk[k]) - float(lr_[k])) <= 2e-2 * abs(float(lr_[k])) + 1e-4, k
    assert _rel(gk, gr) <= 3e-2


def test_call_trace_without_new_ops_is_todays_and_with_them_the_geometric_calls(tmp_path):
    torch.cuda.set_device(0)
    tr_da, _, batch = _trainer(str(tmp_path), "color,translation,cutout")
    tr_geo, _, _ = _trainer(str(tmp_path), FULL)
    tr_off, _, _ = _trainer(str(tmp_path), "")
    for _ in range(2):
        off, _ = _traced_step(tr_off, batch)
        da, n_da = _traced_step(tr_da, batch)
        geo, n_geo = _traced_step(tr_geo, batch)
        today = []
        for c in off:
            if c == "s2e_make_d_input":
                today += ["s2e_diffaug_draw", "s2e_diffaug_means", "s2e_make_d_input_aug"]
            elif c == "s2e_d_input_grad":
                today.append("s2e_d_input_grad_aug")
            else:
                today.append(c)
        assert da == today
        assert not any("geom" in c for c in da)
        want = [{"s2e_diffaug_draw": "s2e_diffaug_draw_geom", "s2e_make_d_input_aug": "s2e_make_d_input_aug_geom",
                 "s2e_d_input_grad_aug": "s2e_d_input_grad_aug_geom"}.get(c, c) for c in today]
        assert geo == want and n_geo == n_da


def test_cuda_graph_replays_draw_like_eager_at_the_same_counters(tmp_path, monkeypatch):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    tr, oopt, batch = _trainer(str(tmp_path), FULL, diff_augment_p=0.5)
    m = tr.pix2pix_model
    drawn, real_draw = [], ops.diffaug_draw_geom

    def spy(*args):
        drawn.append(real_draw(*args))
        return drawn[-1]
    monkeypatch.setattr(ops, "diffaug_draw_geom", spy)
    tr.run_generator_one_step({k: v.clone() for k, v in batch.items()})
    tr.run_discriminator_one_step({k: v.clone() for k, v in batch.items()})
    torch.cuda.synchronize()
    before = m.diffaug_state.tolist()
    tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=2)
    torch.cuda.synchronize()
    assert m.diffaug_state.tolist() == before
    cap_g, cap_d = drawn[-2], drawn[-1]
    replayed = []
    for _ in range(2):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        torch.cuda.synchronize()
        replayed.append([t.clone() for t in cap_g])
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        replayed.append([t.clone() for t in cap_d])
    assert m.diffaug_state.tolist() == [before[0], before[1] + 4]
    B, _, H, W = batch["label"].shape
    st = _state(*before)
    for got in replayed:
        want = real_draw(st, _p(0.5), B, 0, H, W)
        assert all(torch.equal(a, b) for a, b in zip(got, want))
    assert not torch.equal(replayed[0][1], replayed[2][1])
    tr.disable_cuda_graphs()


def test_ada_with_geometric_moves_p_under_cuda_graphs(tmp_path):
    from test_gpu_ada import np_ada
    torch.cuda.set_device(0)
    tr, oopt, batch = _trainer(str(tmp_path), "xflip,geometric", ada_target=0.6, ada_kimg=0.1, ada_interval=2,
                               diff_augment_p=0.5)
    m = tr.pix2pix_model
    for _ in range(2):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
    torch.cuda.synchronize()
    before = {k: v.clone() for k, v in m.ada_state.items()}
    tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=2)
    records, ps = [], []
    for _ in range(10):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        records.append(m.ada_state["record"].cpu().numpy().copy())
        ps.append(float(m.ada_state["p"]))
    acc, pos, p, want = before["acc"].cpu().numpy(), int(before["pos"]), float(before["p"]), []
    for rec in records:
        acc, pos, p = np_ada(acc, pos, p, rec, 0.6, 0.1, 2)
        want.append(p)
    assert ps == want and len(set(ps)) > 1, ps
    tr.disable_cuda_graphs()


# ------------------------------------------------------------------------------------------ two ranks
def _worker(rank, world, port, tmp, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                          LOCAL_RANK=str(rank))
        torch.cuda.set_device(0)
        import torch.distributed as dist
        dist.init_process_group("gloo", timeout=datetime.timedelta(seconds=90), rank=rank, world_size=world)
        from seg2eye_b200 import ops
        from seg2eye_b200.models.pix2pix_model import Pix2PixModel
        from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
        oopt, opt = _opts(tmp, FULL, norm_G="spectralspadesyncbatch3x3")
        opt.gpu_ids = [0]
        torch.manual_seed(100 + rank)
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        m = tr.pix2pix_model
        sds = _sds(oopt, 61)
        _load(m, sds)
        m.train()
        full = O.synth_batch(oopt, 2 * world, 64)
        shard = {k: v[2 * rank:2 * rank + 2].clone() for k, v in full.items()}
        st0 = m.diffaug_state.clone()
        drawn, real_draw = [], ops.diffaug_draw_geom

        def spy(*args):
            drawn.append([t.clone() for t in real_draw(*args)])
            return drawn[-1]
        ops.diffaug_draw_geom = spy
        res = {"state": st0.cpu()}
        if rank == 0:
            with contextlib.redirect_stdout(io.StringIO()):
                mb = Pix2PixModel(_opts(tmp, FULL, norm_G="spectralspadebatch3x3")[1])
            _load(mb, sds)
            mb.diffaug_state.copy_(st0)
            mb.train()
            losses_f, _ = mb({k: v.clone().cuda() for k, v in full.items()}, mode="generator")
            sum(losses_f.values()).mean().backward()
            pB = dict(mb.netG.named_parameters())
            g_full = {n: pB[n].grad.detach().clone() for n in NAMES}
            res["losses_full"] = torch.stack([v.reshape(-1)[0].detach() for v in losses_f.values()]).cpu()
            res["draw_full"] = [t.cpu() for t in drawn[-1]]
            del losses_f, mb
        tr.reducer_G.remove_hooks()
        dist.barrier()
        tr.optimizer_G.zero_grad()
        tr.reducer_G.armed, tr.reducer_D.armed = True, False
        losses, _ = tr._fb("G", {k: v.clone().cuda() for k, v in shard.items()})
        tr.reducer_G.allreduce()
        res["draw"] = [t.cpu() for t in drawn[-1]]
        lsum = torch.stack([v.reshape(-1)[0].detach() for v in losses.values()])
        dist.all_reduce(lsum)
        res["losses_sharded_mean"] = (lsum / world).cpu()
        if rank == 0:
            pG = dict(m.netG.named_parameters())
            res["grad_err"] = {n: _rel(pG[n].grad, g_full[n]) for n in g_full}
        ops.diffaug_draw_geom = real_draw
        torch.cuda.synchronize()
        res = {k: ([t.numpy() for t in v] if isinstance(v, list) else v.numpy() if torch.is_tensor(v) else v)
               for k, v in res.items()}
        q.put((rank, res, None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:      # noqa: BLE001 -- report to the parent instead of hanging it
        import traceback
        q.put((rank, None, traceback.format_exc()))


def test_two_ranks_on_one_gpu_match_full_batch(tmp_path):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(tmp_path), q), daemon=True) for r in range(world)]
    for p in procs:
        p.start()
    got = []
    try:
        for _ in procs:
            got.append(q.get(timeout=400))
            if got[-1][2] is not None:
                break
    finally:
        for p in procs:
            p.join(5 if (got and got[-1][2] is not None) else 60)
            if p.is_alive():
                p.kill()
    for rank, res, err in got:
        assert err is None, "rank %d: %s" % (rank, err)
    res = {rank: r for rank, r, _ in got}
    r0 = res[0]
    print("grad_err %s\nlosses sharded %s full %s" % (r0["grad_err"], r0["losses_sharded_mean"].tolist(),
                                                       r0["losses_full"].tolist()))
    assert all(np.array_equal(r["state"], r0["state"]) for r in res.values())
    for rank, r in res.items():       # records, matrices and masks: what one process draws for samples 2r, 2r + 1
        for a, b in zip(r["draw"], r0["draw_full"]):
            assert a.tobytes() == b[2 * rank:2 * rank + 2].tobytes(), rank
    vals = sorted(r0["grad_err"].values())
    assert vals[len(vals) // 2] < 5e-2 and vals[-1] < 1e-1, r0["grad_err"]
    assert np.allclose(r0["losses_sharded_mean"], r0["losses_full"], rtol=2e-2, atol=2e-2)
