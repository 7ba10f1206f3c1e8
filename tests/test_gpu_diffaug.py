"""`--diff_augment` on the device: the Philox draws against a NumPy restatement, bit for bit; the augmented D-input layout
kernel and its adjoint against a float64 torch restatement; one G step and one D step of the model against the same model
fed the restatement; the C-ABI call trace with the option off and on; draws inside CUDA-graph replays; and two
data-parallel ranks against one process on the whole batch."""
import contextlib
import datetime
import io
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import seg2eye_oracle as O

pytestmark = pytest.mark.gpu

COLOR, TRANSLATION, CUTOUT = 1, 2, 4
POLICIES = {"color": COLOR, "translation": TRANSLATION, "cutout": CUTOUT}
SIZES = {"R1": (320, 256), "R2": (640, 384), "odd": (37, 23)}


# ------------------------------------------------------------------------------------------ NumPy restatement of the RNG
_MASK = np.uint64(0xFFFFFFFF)


def _philox4x32_10(c, key):
    """Philox4x32-10 on arrays of counters: c = 4 uint64 arrays holding 32-bit words, key = two 32-bit ints."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK for x in c]
    k0, k1 = np.uint64(key[0]), np.uint64(key[1])
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _MASK, (k1 + np.uint64(0xBB67AE85)) & _MASK
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
    return c


def _unit(r):
    return ((r >> np.uint64(8)).astype(np.float64) * 2.0 ** -24).astype(np.float32)


def _below(r, n):
    return ((r * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def np_records(seed, counter, offset, B, H, W):
    """The [B, 6] records (u0, u1, tx, ty, ox, oy) the header specifies."""
    s, c = seed % 2 ** 64, counter % 2 ** 64
    key = (s & 0xFFFFFFFF, s >> 32)
    idx = np.arange(offset, offset + B, dtype=np.uint64)
    lo, hi = np.full(B, c & 0xFFFFFFFF, np.uint64), np.full(B, c >> 32, np.uint64)
    r0 = _philox4x32_10([idx, lo, hi, np.zeros(B, np.uint64)], key)
    r1 = _philox4x32_10([idx, lo, hi, np.ones(B, np.uint64)], key)
    sx, sy = int(H / 8 + 0.5), int(W / 8 + 0.5)
    cx, cy = int(H / 2 + 0.5), int(W / 2 + 0.5)
    out = np.stack([_unit(r0[0]), _unit(r0[1]), _below(r0[2], 2 * sx + 1) - sx, _below(r0[3], 2 * sy + 1) - sy,
                    _below(r1[0], H + 1 - cx % 2), _below(r1[1], W + 1 - cy % 2)], 1)
    return out.astype(np.float32)


def _state(seed, counter):
    return torch.tensor([seed, counter], dtype=torch.int64, device="cuda")


def test_numpy_philox_reproduces_the_random123_known_answers():
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(x) for x in _philox4x32_10(ctr, key)) == want


@pytest.mark.parametrize("size", list(SIZES))
def test_draws_match_numpy_philox_bit_for_bit(size):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    H, W = SIZES[size]
    for seed in (0, 1, -1, 0x0123456789ABCDEF, -2 ** 63, 987654321):
        for counter in (0, 1, 77777, 2 ** 32 - 1, 2 ** 32 + 7, 3 * 2 ** 40 + 11):
            for offset, B in ((0, 1), (0, 16), (5, 3), (2 ** 31 + 9, 37), (2 ** 32 - 4, 4)):
                st = _state(seed, counter)
                got = ops.diffaug_draw(st, B, offset, H, W).cpu().numpy()
                want = np_records(seed, counter, offset, B, H, W)
                assert got.tobytes() == want.tobytes(), (seed, counter, offset, B, got, want)
                assert st.tolist() == [seed, counter + 1]         # one step per draw, on the device


def test_draw_reproducible_covers_every_translation_and_is_uniform():
    from scipy import stats
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    H, W = SIZES["R2"]
    st = _state(424242, 5)
    a = ops.diffaug_draw(st, 8, 0, H, W)
    st.copy_(_state(424242, 5))
    b = ops.diffaug_draw(st, 4, 4, H, W)      # same (seed, counter, index) -> same record, whatever the batch split
    assert torch.equal(a[4:], b)
    assert int(st[1]) == 6
    recs = torch.cat([ops.diffaug_draw(st, 4096, 0, H, W) for _ in range(16)]).cpu().numpy()    # 2^16 records
    assert int(st[1]) == 22
    sx, sy = int(H / 8 + 0.5), int(W / 8 + 0.5)
    assert set(recs[:, 2].astype(int)) == set(range(-sx, sx + 1))
    assert set(recs[:, 3].astype(int)) == set(range(-sy, sy + 1))
    cx, cy = int(H / 2 + 0.5), int(W / 2 + 0.5)
    for col, n in ((0, None), (1, None), (4, H + 1 - cx % 2), (5, W + 1 - cy % 2)):
        v = recs[:, col]
        if n is None:
            assert v.min() >= 0 and v.max() < 1
            bins, expected = np.floor(v * 16).astype(int), np.full(16, len(v) / 16)
        else:
            assert v.min() >= 0 and v.max() <= n - 1
            bins = (v.astype(np.int64) * 16) // n
            expected = np.bincount((np.arange(n) * 16) // n, minlength=16) / n * len(v)
        p = stats.chisquare(np.bincount(bins, minlength=16), expected).pvalue
        assert p > 1e-4, (col, p)


# ------------------------------------------------------------------------------------------ float64 restatement
def ref_d_input(seg, fake, real, rec, policy, cpad, means=None):
    """DiffAugment of cat([cat([seg,fake],1), cat([seg,real],1)], 0) in float64 torch, NHWC with cpad channels.  `means`:
    the per-image means to use for contrast ([2B]); None forms them from fake / real (differentiably)."""
    B, nc, H, W = seg.shape
    seg, fake, real = seg.double(), fake.double(), real.double()
    r = torch.cat([rec, rec]).double()
    img = torch.cat([fake, real])[:, 0]
    if policy & COLOR:
        m = img.mean(dim=(1, 2)) if means is None else means.double()
        br, ct = r[:, 0] - 0.5, r[:, 1] + 0.5
        mb = (m + br)[:, None, None]
        img = (img + br[:, None, None] - mb) * ct[:, None, None] + mb
    x = torch.cat([torch.cat([seg, seg]), img[:, None]], 1)                 # (2B, nc + 1, H, W)
    dev = x.device
    ii = torch.arange(H, device=dev)[None, :, None].expand(2 * B, H, W)
    jj = torch.arange(W, device=dev)[None, None, :].expand(2 * B, H, W)
    keep = torch.ones(2 * B, H, W, dtype=torch.bool, device=dev)
    si, sj = ii, jj
    if policy & TRANSLATION:
        si, sj = ii + r[:, 2].long()[:, None, None], jj + r[:, 3].long()[:, None, None]
        keep &= (si >= 0) & (si < H) & (sj >= 0) & (sj < W)
    if policy & CUTOUT:
        cx, cy = int(H / 2 + 0.5), int(W / 2 + 0.5)
        x0, y0 = (r[:, 4].long() - cx // 2)[:, None, None], (r[:, 5].long() - cy // 2)[:, None, None]
        keep &= ~((ii >= x0) & (ii < x0 + cx) & (jj >= y0) & (jj < y0 + cy))
    bb = torch.arange(2 * B, device=dev)[:, None, None].expand(2 * B, H, W)
    g = x.permute(0, 2, 3, 1)[bb, si.clamp(0, H - 1), sj.clamp(0, W - 1)]  # (2B, H, W, nc + 1)
    out = g * keep[..., None]
    return torch.nn.functional.pad(out, (0, cpad - (nc + 1)))


def _inputs(B, nc, H, W, seed):
    gen = torch.Generator().manual_seed(seed)
    lab = torch.randint(0, nc, (B, H, W), generator=gen)
    seg = torch.nn.functional.one_hot(lab, nc).permute(0, 3, 1, 2).float()
    fake = torch.rand(B, 1, H, W, generator=gen) * 2 - 1
    real = torch.rand(B, 1, H, W, generator=gen) * 1.6 - 0.7
    return seg.cuda(), fake.cuda(), real.cuda()


CASES = [(1, 4, 37, 23), (3, 4, 64, 40), (3, 35, 33, 47), (1, 35, 20, 31)]
FWD_POLICIES = ["translation", "cutout", "translation,cutout", "color", "color,translation,cutout"]


def _bits(policy):
    return sum(POLICIES[p] for p in policy.split(","))


def _means(fake, real):
    from seg2eye_b200 import _lib as L
    B, _, H, W = fake.shape
    m = torch.empty(2 * B, device="cuda")
    L.call("s2e_diffaug_means", L.ptr(fake), L.ptr(real), B, H, W, L.ptr(m), L.stream())
    return m


def _bf16_ulp(v):
    a = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


@pytest.mark.parametrize("policy", FWD_POLICIES)
@pytest.mark.parametrize("case", CASES)
def test_forward_matches_float64_restatement(case, policy):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    bits = _bits(policy)
    seg, fake, real = _inputs(B, nc, H, W, 3 + B + nc)
    cpad = -(-(nc + 1) // 16) * 16
    st = _state(1234 + nc, 9)
    for _ in range(3):       # several draws: different shifts and rectangles
        rec = ops.diffaug_draw(st, B, 0, H, W)
        out = ops.MakeDInputAugFn.apply(seg, fake, real, cpad, rec, bits)
        torch.cuda.synchronize()
        assert out.shape == (2 * B, H, W, cpad) and out.dtype == torch.bfloat16
        assert torch.all(out[..., nc + 1:] == 0)                              # padding channels
        means = _means(fake, real)
        ref = ref_d_input(seg, fake, real, rec, bits, cpad, means)
        if bits & COLOR:
            # the image channel within one bf16 ulp (fp32 arithmetic in the kernel), the segmap channels bitwise
            assert torch.equal(out[..., :nc], ref[..., :nc].to(torch.bfloat16))
            d = (out[..., nc].double() - ref[..., nc]).abs()
            ulp = torch.maximum(_bf16_ulp(ref[..., nc]), _bf16_ulp(out[..., nc].double()))
            assert torch.all(d <= ulp), float((d / ulp).max())
            full = torch.tensor([fake[b].double().mean() for b in range(B)] + [real[b].double().mean() for b in range(B)])
            assert torch.allclose(means.double().cpu(), full, rtol=0, atol=1e-6)
        else:
            assert torch.equal(out, ref.to(torch.bfloat16))
        # rows b and B + b share the record: with fake == real they are identical
        same = ops.MakeDInputAugFn.apply(seg, real, real, cpad, rec, bits)
        assert torch.equal(same[:B], same[B:])
    assert torch.equal(out, ops.MakeDInputAugFn.apply(seg, fake, real, cpad, rec, bits))   # deterministic


@pytest.mark.parametrize("policy", FWD_POLICIES)
@pytest.mark.parametrize("case", CASES)
def test_backward_matches_float64_autograd_and_is_the_adjoint(case, policy):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    bits = _bits(policy)
    seg, fake, real = _inputs(B, nc, H, W, 17 + B)
    cpad = -(-(nc + 1) // 16) * 16
    rec = ops.diffaug_draw(_state(99 + nc, 2 ** 32 + 1), B, 0, H, W)
    gen = torch.Generator().manual_seed(5)
    g = (torch.randn(2 * B, H, W, cpad, generator=gen)).to(torch.bfloat16).cuda()
    f = fake.clone().requires_grad_(True)
    ops.MakeDInputAugFn.apply(seg, f, real, cpad, rec, bits).backward(g)
    got = f.grad.double()
    f64 = fake.double().requires_grad_(True)
    (ref_d_input(seg, f64, real, rec, bits, cpad) * g.double()).sum().backward()
    want = f64.grad
    if bits & COLOR:
        # dfake = c g' + (1 - c) mean(g'): fp64 sums, then a few fp32 roundings (c = u1 + 0.5 itself rounds in fp32)
        f0 = torch.zeros_like(fake.double()).requires_grad_(True)
        (ref_d_input(seg, f0, real, rec, bits & ~COLOR, cpad) * g.double()).sum().backward()
        gp = f0.grad       # g', the gathered gradient
        c = (rec[:, 1].double() + 0.5).view(B, 1, 1, 1)
        mean = gp.mean(dim=(1, 2, 3), keepdim=True).abs()
        bound = 2.0 ** -21 * (c * gp.abs() + ((1 - c).abs() + 1) * mean) + 1e-30
        assert torch.all((got - want).abs() <= bound), float(((got - want).abs() / bound).max())
    else:
        assert torch.equal(got, want)
    # <T x, g> == <x, T^T g> in float64, T the linear part of the map fake -> output (brightness is a constant shift)
    x = torch.randn(B, 1, H, W, generator=gen, dtype=torch.float64).cuda()
    zero = torch.zeros_like(real)
    tx = ref_d_input(seg, x, zero, rec, bits, cpad) - ref_d_input(seg, torch.zeros_like(x), zero, rec, bits, cpad)
    lhs = float((tx[:B, ..., nc] * g[:B, ..., nc].double()).sum())
    rhs = float((x * got).sum())
    assert abs(lhs - rhs) <= (1e-6 if bits & COLOR else 1e-12) * float((x.abs() * got.abs()).sum()), (lhs, rhs)


# ------------------------------------------------------------------------------------------ model and trainer
def _opts(tmp, policy, ngf=16, **kw):
    o = O.make_opt(ngf=ngf, ndf=16, lambda_l1=10.0, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[0], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=tmp, name="da", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale",
             diff_augment=policy)
    return o, SimpleNamespace(**d)


def _sds(oopt, seed):
    return dict(G=O.synth_state(O.generator_shapes(oopt), seed), D=O.synth_state(O.discriminator_shapes(oopt), seed + 1),
                E=O.synth_state(O.encoder_shapes(oopt), seed + 2))


def _load(m, sds):
    for net, k in ((m.netG, "G"), (m.netD, "D"), (m.netE, "E")):
        net.load_state_dict({a: b.clone() for a, b in sds[k].items()})


def _trainer(tmp, policy, seed=31, **kw):
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    oopt, opt = _opts(tmp, policy, **kw)
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    _load(tr.pix2pix_model, _sds(oopt, seed))
    return tr, oopt, O.synth_batch(oopt, 2, seed + 3)


class _RestatedDInput:
    """Stands in for ops.MakeDInputAugFn: the float64 restatement, rounded to bf16, with torch autograd to the fake."""

    @staticmethod
    def apply(seg, fake, real, cpad, params, policy):
        return ref_d_input(seg, fake, real, params, policy, max(cpad, seg.shape[1] + 1)).to(torch.bfloat16).contiguous()


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("no_ganFeat_loss", [False, True])
def test_model_steps_match_the_restated_d_input(tmp_path, monkeypatch, no_ganFeat_loss):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    torch.cuda.set_device(0)
    oopt, opt = _opts(str(tmp_path), "color,translation,cutout", no_ganFeat_loss=no_ganFeat_loss)
    sds = _sds(oopt, 41)
    batch = O.synth_batch(oopt, 3, 44)
    res = {}
    for name in ("kernel", "restated"):
        with contextlib.redirect_stdout(io.StringIO()):
            m = Pix2PixModel(opt)
        _load(m, sds)
        m.diffaug_state.copy_(_state(2024, 3))
        m.train()
        with monkeypatch.context() as mp_:
            if name == "restated":
                mp_.setattr(ops, "MakeDInputAugFn", _RestatedDInput)
            losses, fake = m({k: v.clone() for k, v in batch.items()}, mode="generator")
            fake.retain_grad()
            sum(losses.values()).mean().backward()
            d_losses = m({k: v.clone() for k, v in batch.items()}, mode="discriminator")
        torch.cuda.synchronize()
        res[name] = ({k: v.detach().reshape(-1)[0] for k, v in {**losses, **d_losses}.items()}, fake.grad.detach().clone(),
                     m.diffaug_state.tolist())
    (lk, gk, sk), (lr_, gr, sr) = res["kernel"], res["restated"]
    assert sk == sr == [2024, 5]           # one draw in the G step, one in the D step
    assert set(lk) == set(lr_) and ("GAN_Feat" in lk) == (not no_ganFeat_loss)
    print("losses kernel %s restated %s, dfake rel %.2e" % ({k: float(v) for k, v in lk.items()},
                                                           {k: float(v) for k, v in lr_.items()}, _rel(gk, gr)))
    for k in lk:    # tests/test_gpu_modules.py TOL_LOSS; TOL_PAIR for the image gradient
        assert abs(float(lk[k]) - float(lr_[k])) <= 2e-2 * abs(float(lr_[k])) + 1e-4, k
    assert _rel(gk, gr) <= 3e-2


def _traced_step(tr, batch):
    from seg2eye_b200 import _lib as L
    calls, real = [], L.call

    def rec(name, *args):
        calls.append(name)
        return real(name, *args)
    L.call = rec
    n0 = L.launches
    try:
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
    finally:
        L.call = real
    return calls, L.launches - n0


NEW_CALLS = {"s2e_diffaug_draw", "s2e_diffaug_means", "s2e_make_d_input_aug", "s2e_d_input_grad_aug"}


@pytest.mark.parametrize("policy", ["color,translation,cutout", "translation"])
def test_policy_off_runs_todays_calls_and_on_adds_the_new_ones(tmp_path, policy):
    torch.cuda.set_device(0)
    tr_off, _, batch = _trainer(str(tmp_path), "")
    tr_on, _, _ = _trainer(str(tmp_path), policy)
    color = "color" in policy
    for _ in range(2):
        off, n_off = _traced_step(tr_off, batch)
        on, n_on = _traced_step(tr_on, batch)
        assert not NEW_CALLS & set(off)
        assert off.count("s2e_make_d_input") == 2 and off.count("s2e_d_input_grad") == 1
        want = []
        for c in off:
            if c == "s2e_make_d_input":
                want += ["s2e_diffaug_draw"] + (["s2e_diffaug_means"] if color else []) + ["s2e_make_d_input_aug"]
            elif c == "s2e_d_input_grad":
                want.append("s2e_d_input_grad_aug")
            else:
                want.append(c)
        assert on == want
        assert n_on == n_off + (4 if color else 2)


def test_cuda_graph_replays_draw_like_eager_at_the_same_counters(tmp_path, monkeypatch):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    tr, oopt, batch = _trainer(str(tmp_path), "color,translation,cutout")
    m = tr.pix2pix_model
    drawn, real_draw = [], ops.diffaug_draw

    def spy(*args):
        drawn.append(real_draw(*args))
        return drawn[-1]
    monkeypatch.setattr(ops, "diffaug_draw", spy)
    tr.run_generator_one_step({k: v.clone() for k, v in batch.items()})      # eager steps first, like a real run
    tr.run_discriminator_one_step({k: v.clone() for k, v in batch.items()})
    torch.cuda.synchronize()
    before = m.diffaug_state.tolist()
    assert before[1] == 2
    tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=2)
    torch.cuda.synchronize()
    assert m.diffaug_state.tolist() == before, "enable_cuda_graphs moved the draw counter"
    rec_g, rec_d = drawn[-2], drawn[-1]       # the captured G step's and D step's record buffers
    replayed = []
    for _ in range(2):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        torch.cuda.synchronize()
        replayed.append(rec_g.clone())
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        replayed.append(rec_d.clone())
    assert m.diffaug_state.tolist() == [before[0], before[1] + 4]
    B, _, H, W = batch["label"].shape
    st = _state(*before)
    eager = [real_draw(st, B, 0, H, W) for _ in range(4)]
    for a, b in zip(replayed, eager):
        assert torch.equal(a, b)
    assert not torch.equal(replayed[0], replayed[2]) and not torch.equal(replayed[0], replayed[1])
    tr.disable_cuda_graphs()


# ------------------------------------------------------------------------------------------ two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


NAMES = ["fc.weight", "head_0.conv_0.weight_orig", "up_1.norm_0.spade.mlp_gamma.weight", "up_3.conv_1.weight_orig",
         "up_3.norm_1.adain.linear.weight", "conv_img.weight", "head_0.norm_0.spade.mlp_shared.0.weight"]


def _worker(rank, world, port, tmp, q, backend):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                          LOCAL_RANK=str(rank))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        import torch.distributed as dist
        kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
        dist.init_process_group(backend, timeout=datetime.timedelta(seconds=90), rank=rank, world_size=world, **kw)
        from seg2eye_b200 import ops
        from seg2eye_b200.models.pix2pix_model import Pix2PixModel
        from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
        policy = "color,translation,cutout"
        oopt, opt = _opts(tmp, policy, norm_G="spectralspadesyncbatch3x3")
        opt.gpu_ids = [dev]
        torch.manual_seed(100 + rank)      # a different seed per rank: the broadcast must align them
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        m = tr.pix2pix_model
        sds = _sds(oopt, 71)
        _load(m, sds)
        m.train()
        full = O.synth_batch(oopt, 2 * world, 74)
        shard = {k: v[2 * rank:2 * rank + 2].clone() for k, v in full.items()}
        st0 = m.diffaug_state.clone()
        drawn, real_draw = [], ops.diffaug_draw

        def spy(*args):
            drawn.append(real_draw(*args).clone())
            return drawn[-1]
        ops.diffaug_draw = spy
        res = {"state": st0.cpu()}
        if rank == 0:     # one process, the whole batch, the same weights and generator state
            with contextlib.redirect_stdout(io.StringIO()):
                mb = Pix2PixModel(_opts(tmp, policy, norm_G="spectralspadebatch3x3")[1])
            _load(mb, sds)
            mb.diffaug_state.copy_(st0)
            mb.train()
            losses_f, _ = mb({k: v.clone().cuda() for k, v in full.items()}, mode="generator")
            sum(losses_f.values()).mean().backward()
            pB = dict(mb.netG.named_parameters())
            g_full = {n: pB[n].grad.detach().clone() for n in NAMES}
            res["losses_full"] = torch.stack([v.reshape(-1)[0].detach() for v in losses_f.values()]).cpu()
            res["records_full"] = drawn[-1].cpu()
            del losses_f, mb
        tr.reducer_G.remove_hooks()
        dist.barrier()
        tr.optimizer_G.zero_grad()
        tr.reducer_G.armed, tr.reducer_D.armed = True, False
        losses, _ = tr._fb("G", {k: v.clone().cuda() for k, v in shard.items()})
        tr.reducer_G.allreduce()
        res["records"] = drawn[-1].cpu()
        lsum = torch.stack([v.reshape(-1)[0].detach() for v in losses.values()])
        dist.all_reduce(lsum)
        res["losses_sharded_mean"] = (lsum / world).cpu()
        if rank == 0:
            pG = dict(m.netG.named_parameters())
            res["grad_err"] = {n: _rel(pG[n].grad, g_full[n]) for n in NAMES}
        ops.diffaug_draw = real_draw
        torch.cuda.synchronize()
        # plain arrays: a tensor sent through the queue would be shared by a file descriptor of this (exiting) process
        res = {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in res.items()}
        q.put((rank, res, None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:      # noqa: BLE001 -- report to the parent instead of hanging it
        import traceback
        q.put((rank, None, traceback.format_exc()))


def _run(tmp, backend, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, tmp, q, backend), daemon=True) for r in range(world)]
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
    assert len(got) == world
    res = {rank: {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in r.items()} for rank, r, _ in got}
    r0 = res[0]
    print("grad_err %s\nlosses sharded %s full %s" % (r0["grad_err"], r0["losses_sharded_mean"].tolist(),
                                                       r0["losses_full"].tolist()))
    assert all(torch.equal(r["state"], r0["state"]) for r in res.values())    # rank 0's seed everywhere
    for rank, r in res.items():       # rank r draws what one process draws for the global samples 2r, 2r + 1
        assert torch.equal(r["records"], r0["records_full"][2 * rank:2 * rank + 2]), rank
    vals = sorted(r0["grad_err"].values())      # tests/test_gpu_syncbn.py::test_two_ranks_on_one_gpu_match_full_batch
    assert vals[len(vals) // 2] < 5e-2 and vals[-1] < 1e-1, r0["grad_err"]
    assert torch.allclose(r0["losses_sharded_mean"], r0["losses_full"], rtol=2e-2, atol=2e-2)


def test_two_ranks_on_one_gpu_match_full_batch(tmp_path):
    """gloo, both ranks on GPU 0, eager, --norm_G spectralspadesyncbatch3x3 with every op on."""
    _run(str(tmp_path), "gloo")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpus_match_full_batch(tmp_path):
    _run(str(tmp_path), "nccl")
