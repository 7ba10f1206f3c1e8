"""`--diff_augment_p` / `--ada_target` on the device: the gated draws against a NumPy restatement, bit for bit; the masked
D-input kernels against the unmasked ones (full mask), today's layout kernels (empty mask) and a float64 restatement per
sample (mixed masks); the real-half sign sums of the logit head and of S2E_RED_SIGN; the controller against a NumPy fp64
recurrence; the model's records and p trajectory, eager and under CUDA graphs; the C-ABI call trace; and two ranks."""
import contextlib
import datetime
import io
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import seg2eye_oracle as O
from test_gpu_diffaug import (COLOR, CUTOUT, TRANSLATION, _bf16_ulp, _free_port, _inputs, _means, _opts, _philox4x32_10,
                              _sds, _load, _state, _traced_step, _trainer, _unit, np_records, ref_d_input)

pytestmark = pytest.mark.gpu

P_VALUES = (0.0, 2.0 ** -24, 0.3, 0.5, 1 - 2.0 ** -24, 1.0)


def np_opmask(seed, counter, offset, B, p):
    """opmask[b]: COLOR iff unit(r6) < p, TRANSLATION iff unit(r7) < p, CUTOUT iff unit(r8) < p (fp64 comparison), r6, r7 =
    block 1's words 2, 3 and r8 = block 2's word 0 of the record's Philox counter."""
    s, c = seed % 2 ** 64, counter % 2 ** 64
    key = (s & 0xFFFFFFFF, s >> 32)
    idx = np.arange(offset, offset + B, dtype=np.uint64)
    lo, hi = np.full(B, c & 0xFFFFFFFF, np.uint64), np.full(B, c >> 32, np.uint64)
    r1 = _philox4x32_10([idx, lo, hi, np.ones(B, np.uint64)], key)
    r2 = _philox4x32_10([idx, lo, hi, np.full(B, 2, np.uint64)], key)
    gate = lambda r: _unit(r).astype(np.float64) < p     # noqa: E731
    return (gate(r1[2]) * COLOR | gate(r1[3]) * TRANSLATION | gate(r2[0]) * CUTOUT).astype(np.int32)


def _p(v):
    return torch.tensor([v], dtype=torch.float64, device="cuda")


# ------------------------------------------------------------------------------------------ draws
def test_gated_draw_keeps_the_records_and_matches_numpy_gates_bit_for_bit():
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    H, W = 640, 384
    for seed in (0, -1, 0x0123456789ABCDEF, 987654321):
        for counter in (0, 77777, 2 ** 32 + 7, 3 * 2 ** 40 + 11):
            for offset, B in ((0, 16), (5, 3), (2 ** 31 + 9, 37), (2 ** 32 - 4, 4)):
                for p in P_VALUES:
                    st_a, st_b = _state(seed, counter), _state(seed, counter)
                    rec_a = ops.diffaug_draw(st_a, B, offset, H, W)
                    rec_b, mask = ops.diffaug_draw_p(st_b, _p(p), B, offset, H, W)
                    assert rec_b.cpu().numpy().tobytes() == rec_a.cpu().numpy().tobytes()
                    assert rec_b.cpu().numpy().tobytes() == np_records(seed, counter, offset, B, H, W).tobytes()
                    assert st_a.tolist() == st_b.tolist() == [seed, counter + 1]
                    want = np_opmask(seed, counter, offset, B, p)
                    assert np.array_equal(mask.cpu().numpy(), want), (seed, counter, offset, p)
                    if p == 0.0:
                        assert not want.any()
                    if p == 1.0:
                        assert (want == 7).all()


def test_gates_have_the_probability_and_are_pairwise_independent():
    from scipy import stats
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    p, n = 0.3, 1 << 14
    st = _state(20201207, 3)
    masks = torch.cat([ops.diffaug_draw_p(st, _p(p), 4096, 0, 64, 64)[1] for _ in range(n // 4096)]).cpu().numpy()
    bits = {k: (masks & k) != 0 for k in (COLOR, TRANSLATION, CUTOUT)}
    sd = (n * p * (1 - p)) ** 0.5
    for k, g in bits.items():      # a deterministic 5-sigma binomial bound: the seed is fixed
        assert abs(int(g.sum()) - n * p) <= 5 * sd, (k, int(g.sum()))
    for a, b in ((COLOR, TRANSLATION), (COLOR, CUTOUT), (TRANSLATION, CUTOUT)):
        table = np.array([[np.sum(bits[a] & bits[b]), np.sum(bits[a] & ~bits[b])],
                          [np.sum(~bits[a] & bits[b]), np.sum(~bits[a] & ~bits[b])]])
        assert stats.chi2_contingency(table).pvalue > 1e-4, (a, b, table)


# ------------------------------------------------------------------------------------------ masked kernels
CASES = [(8, 4, 37, 23), (8, 35, 33, 47)]
ALL = COLOR | TRANSLATION | CUTOUT


@pytest.mark.parametrize("case", CASES)
def test_masked_kernels_at_full_and_empty_masks_equal_todays_kernels(case):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    seg, fake, real = _inputs(B, nc, H, W, 11 + nc)
    cpad = -(-(nc + 1) // 16) * 16
    rec = ops.diffaug_draw(_state(5 + nc, 1), B, 0, H, W)
    g = torch.randn(2 * B, H, W, cpad, generator=torch.Generator().manual_seed(2)).to(torch.bfloat16).cuda()
    for policy in (ALL, TRANSLATION | CUTOUT, COLOR):
        full = torch.full((B,), 7, dtype=torch.int32, device="cuda")
        f1, f2 = fake.clone().requires_grad_(True), fake.clone().requires_grad_(True)
        a = ops.MakeDInputAugFn.apply(seg, f1, real, cpad, rec, policy)
        b = ops.MakeDInputAugMaskedFn.apply(seg, f2, real, cpad, rec, full, policy)
        a.backward(g)
        b.backward(g)
        assert torch.equal(a, b) and torch.equal(f1.grad, f2.grad), policy
        empty = torch.zeros(B, dtype=torch.int32, device="cuda")
        f1, f2 = fake.clone().requires_grad_(True), fake.clone().requires_grad_(True)
        a = ops.MakeDInputFn.apply(seg, f1, real, cpad)
        b = ops.MakeDInputAugMaskedFn.apply(seg, f2, real, cpad, rec, empty, policy)
        a.backward(g)
        b.backward(g)
        assert torch.equal(a, b) and torch.equal(f1.grad, f2.grad), policy


@pytest.mark.parametrize("case", CASES)
def test_masked_kernels_match_float64_per_sample_and_are_adjoint(case):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, nc, H, W = case
    seg, fake, real = _inputs(B, nc, H, W, 23 + nc)
    cpad = -(-(nc + 1) // 16) * 16
    rec = ops.diffaug_draw(_state(77 + nc, 2 ** 32 + 3), B, 0, H, W)
    mask = torch.arange(B, dtype=torch.int32, device="cuda") % 8            # every gate combination
    gen = torch.Generator().manual_seed(9)
    g = torch.randn(2 * B, H, W, cpad, generator=gen).to(torch.bfloat16).cuda()
    for policy in (ALL, TRANSLATION | CUTOUT, COLOR | CUTOUT):
        f = fake.clone().requires_grad_(True)
        out = ops.MakeDInputAugMaskedFn.apply(seg, f, real, cpad, rec, mask, policy)
        out.backward(g)
        means = _means(fake, real)
        for b in range(B):
            pol = policy & int(mask[b])
            rows = [b, B + b]
            ref = ref_d_input(seg[b:b + 1], fake[b:b + 1], real[b:b + 1], rec[b:b + 1], pol, cpad, means[rows])
            got = out[rows]
            f64 = fake[b:b + 1].double().requires_grad_(True)
            (ref_d_input(seg[b:b + 1], f64, real[b:b + 1], rec[b:b + 1], pol, cpad) * g[rows].double()).sum().backward()
            dgot, dwant = f.grad[b:b + 1].double(), f64.grad
            if pol & COLOR:
                assert torch.equal(got[..., :nc], ref[..., :nc].to(torch.bfloat16))
                d = (got[..., nc].double() - ref[..., nc]).abs()
                assert torch.all(d <= torch.maximum(_bf16_ulp(ref[..., nc]), _bf16_ulp(got[..., nc].double()))), (b, pol)
                f0 = torch.zeros_like(f64).requires_grad_(True)
                (ref_d_input(seg[b:b + 1], f0, real[b:b + 1], rec[b:b + 1], pol & ~COLOR, cpad) * g[rows].double()).sum().backward()
                gp = f0.grad
                c = float(rec[b, 1]) + 0.5
                bound = 2.0 ** -21 * (c * gp.abs() + (abs(1 - c) + 1) * gp.mean().abs()) + 1e-30
                assert torch.all((dgot - dwant).abs() <= bound), (b, pol)
            else:     # no colour: a gather, bitwise both ways
                assert torch.equal(got, ref.to(torch.bfloat16)), (b, pol)
                assert torch.equal(dgot, dwant), (b, pol)
        x = torch.randn(B, 1, H, W, generator=gen, dtype=torch.float64).cuda()
        zero = torch.zeros_like(real)
        lhs = 0.0
        for b in range(B):
            pol = policy & int(mask[b])
            args = (seg[b:b + 1], zero[b:b + 1], rec[b:b + 1], pol, cpad)
            tx = ref_d_input(seg[b:b + 1], x[b:b + 1], *args[1:]) - ref_d_input(seg[b:b + 1], torch.zeros_like(x[b:b + 1]), *args[1:])
            lhs += float((tx[0, ..., nc] * g[b, ..., nc].double()).sum())
        rhs = float((x * f.grad.double()).sum())
        assert abs(lhs - rhs) <= 1e-6 * float((x.abs() * f.grad.double().abs()).sum()), (lhs, rhs)


# ------------------------------------------------------------------------------------------ sign sums
@pytest.mark.parametrize("hw", [(42, 34), (22, 18)])       # the logit maps of D's two scales at 320 x 256
def test_head_sign_slot_is_the_exact_sign_sum_of_the_real_logits(hw):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.networks.layers import Conv2d
    torch.cuda.set_device(0)
    gen = torch.Generator().manual_seed(hw[0])
    conv = Conv2d(128, 1, 4, stride=1, padding=2).cuda()
    B = 4
    x = (torch.randn(2 * B, hw[0] - 1, hw[1] - 1, 128, generator=gen) * 0.3).to(torch.bfloat16).cuda()
    with torch.no_grad():
        y0 = conv.forward_nhwc(x)
        with ops.head_sign_sums() as signs:
            y1 = conv.forward_nhwc(x)
    assert torch.equal(y0, y1) and list(signs) == [y1.data_ptr()] and y1._s2e_gan_sums.shape == (7,)
    want = torch.sign(y1[B:].float()).sum()
    assert float(signs[y1.data_ptr()]) == float(want)
    assert float(ops.sign_sum(y1[B:])) == float(want)                   # S2E_RED_SIGN
    assert abs(float(want)) < y1[B:].numel()                           # both signs occur
    z = torch.tensor([0.0, -0.0, 1.5, -2.0, 3e-38, -1e30, 0.25] * 1001, dtype=torch.bfloat16, device="cuda")
    assert float(ops.sign_sum(z)) == float(torch.sign(z.float()).sum())


@pytest.mark.parametrize("hw", [(41, 33), (21, 17)])
def test_gan_sum_slots_are_unchanged_by_the_sign_slot(hw):
    """Integer tap products (D in {-1, 0, 1}): every logit and every partial sum is an exact integer, so the six GAN sums do
    not depend on the order of the atomics and must be bitwise those of s2e_head_gather, and zero logits occur."""
    from seg2eye_b200 import _lib as L
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    B, (Hi, Wi) = 4, hw
    cfg = ops.ConvCfg(4, 4, 1, 2, L.ACT_NONE)
    Ho, Wo = ops.conv_out_hw(cfg, Hi, Wi)
    desc = ops._desc(2 * B, Hi, Wi, 128, Ho, Wo, 1, ops.conv_taps(cfg), L.ACT_NONE)
    D = torch.randint(-1, 2, (2 * B * Hi * Wi, 16), generator=torch.Generator().manual_seed(Hi)).float().cuda()
    y0, y1 = (torch.empty(2 * B, Ho, Wo, 1, dtype=torch.bfloat16, device="cuda") for _ in range(2))
    s0, s1 = torch.zeros(6, device="cuda"), torch.zeros(7, device="cuda")
    L.call("s2e_head_gather", desc, L.ptr(D), None, None, L.ptr(y0), L.ptr(s0), L.stream())
    L.call("s2e_head_gather_signs", desc, L.ptr(D), None, None, L.ptr(y1), L.ptr(s1), L.ptr(s1[6:]), L.stream())
    assert torch.equal(y0, y1)
    assert s0.cpu().numpy().tobytes() == s1[:6].cpu().numpy().tobytes()
    y = y1.double()
    want = [y[:B].sum(), (y[:B] - 1).clamp(max=0).sum(), (-y[:B] - 1).clamp(max=0).sum(),
            y[B:].sum(), (y[B:] - 1).clamp(max=0).sum(), (-y[B:] - 1).clamp(max=0).sum(), torch.sign(y[B:]).sum()]
    assert s1.cpu().tolist() == [float(w) for w in want]
    assert int((y[B:] == 0).sum()) > 0


# ------------------------------------------------------------------------------------------ controller
def np_ada(acc, pos, p, rec, target, kimg, interval):
    n_d = (len(rec) - 1) // 2
    acc = acc.copy()
    acc[:len(rec)] += rec
    pos += 1
    if pos >= interval:
        r = 0.0
        for i in range(n_d):
            r += acc[2 * i] / acc[2 * i + 1]
        r /= n_d
        sgn = float(r > target) - float(r < target)
        p = min(max(p + sgn * acc[2 * n_d] / (kimg * 1000.0), 0.0), 1.0)
        acc[:len(rec)] = 0.0
        acc[-1] = r
        pos = 0
    return acc, pos, p


def _ada_state(n_d, p):
    n = 2 * n_d + 1
    return {"p": _p(p), "acc": torch.zeros(n + 1, dtype=torch.float64, device="cuda"),
            "pos": torch.zeros(1, dtype=torch.int32, device="cuda"), "record": torch.zeros(n, dtype=torch.float64, device="cuda")}


@pytest.mark.parametrize("interval", [1, 4])
def test_controller_matches_numpy_fp64_recurrence_bit_for_bit(interval):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    rng = np.random.default_rng(interval)
    for n_d, target, kimg, p0 in ((2, 0.6, 0.5, 0.0), (2, 0.5, 0.013, 0.97), (1, 0.3, 500.0, 0.4), (3, 0.6, 0.02, 0.01)):
        st = _ada_state(n_d, p0)
        acc, pos, p = np.zeros(2 * n_d + 2), 0, p0
        N = rng.integers(100, 3000, n_d).astype(np.float64)
        for step in range(40):
            kind = step % 5
            if kind == 0:
                S = N.copy()                       # r = 1 > target
            elif kind == 1:
                S = -N                             # r = -1 < target
            elif kind == 2 and target == 0.5:
                S = N / 2                          # r == target exactly: p stays
            else:
                S = np.floor(rng.uniform(-1, 1, n_d) * N)
            rec = np.empty(2 * n_d + 1)
            rec[0:-1:2], rec[1:-1:2], rec[-1] = S, N, float(rng.integers(1, 64))
            st["record"].copy_(torch.from_numpy(rec))
            ops.ada_update(st, target, kimg, interval)
            acc, pos, p = np_ada(acc, pos, p, rec, target, kimg, interval)
            torch.cuda.synchronize()
            assert st["p"].cpu().numpy().tobytes() == np.array([p]).tobytes(), (n_d, step)
            assert st["acc"].cpu().numpy().tobytes() == acc.tobytes(), (n_d, step)
            assert int(st["pos"]) == pos
    # clamping: a huge step goes to 1 and back to 0, not beyond
    st = _ada_state(1, 0.5)
    for S, want in ((10.0, 1.0), (-10.0, 0.0)):
        st["record"].copy_(torch.tensor([S, 10.0, 1e6], dtype=torch.float64))
        for _ in range(interval):
            ops.ada_update(st, 0.6, 0.001, interval)
        assert float(st["p"]) == want


# ------------------------------------------------------------------------------------------ model
ADA = dict(ada_target=0.6, ada_kimg=0.1, ada_interval=2, diff_augment_p=0.5)     # p moves by 0.04 per update at B2


def _np_trajectory(records, p0, interval, target=0.6, kimg=0.1):
    acc, pos, p, ps = np.zeros(len(records[0]) + 1), 0, p0, []
    for rec in records:
        acc, pos, p = np_ada(acc, pos, p, rec, target, kimg, interval)
        ps.append(p)
    return ps, acc, pos


def _logit_spy(m):
    seen, real_record = [], m._ada_record

    def spy(d_out, signs):
        seen.append([scale[-1].detach() for scale in d_out])    # no autograd graph kept across steps
        return real_record(d_out, signs)
    m._ada_record = spy
    return seen


def _check_record(rec, logits, B):
    for i, y in enumerate(logits):
        real = y[y.shape[0] // 2:]
        assert rec[2 * i] == float(torch.sign(real.float()).sum()) and rec[2 * i + 1] == real.numel(), i
    assert rec[-1] == B


@pytest.mark.parametrize("head", ["gather", "fallback"])
def test_model_records_and_p_trajectory_eager(tmp_path, monkeypatch, head):
    from seg2eye_b200 import ops
    torch.cuda.set_device(0)
    if head == "fallback":      # logits from the tensor-core convolution: S2E_RED_SIGN sums their signs
        monkeypatch.setattr(ops, "HEAD_ON_TC", True)
    tr, oopt, batch = _trainer(str(tmp_path), "color,translation,cutout", **ADA)
    m = tr.pix2pix_model
    assert float(m.ada_state["p"]) == 0.5 and m.ada_interval == 2
    seen = _logit_spy(m)
    calls = []
    real_call = ops.L.call
    monkeypatch.setattr(ops.L, "call", lambda name, *a: (calls.append(name), real_call(name, *a))[1])
    records, ps = [], []
    for _ in range(12):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        records.append(m.ada_state["record"].cpu().numpy().copy())
        _check_record(records[-1], seen[-1], batch["label"].shape[0])
        ps.append(float(m.ada_state["p"]))
    assert ("s2e_head_gather_signs" in calls) == (head == "gather")
    want, acc, pos = _np_trajectory(records, 0.5, 2)
    assert ps == want and len(set(ps)) > 1, ps
    assert m.ada_state["acc"].cpu().numpy().tobytes() == acc.tobytes() and int(m.ada_state["pos"]) == pos
    log = tr.get_latest_losses(include_log_losses=True)
    assert "ada/p" in log and "ada/rt" in log and "ada/p" not in tr.d_losses
    assert abs(float(log["ada/p"]) - ps[-1]) <= 1e-12 and abs(float(log["ada/rt"]) - acc[-1]) <= 1e-12


def test_model_records_and_p_trajectory_under_cuda_graphs(tmp_path):
    torch.cuda.set_device(0)
    tr, oopt, batch = _trainer(str(tmp_path), "color,translation,cutout", **ADA)
    m = tr.pix2pix_model
    seen = _logit_spy(m)
    for _ in range(3):        # eager steps first, like a real run: p has moved off 0 by the capture
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
    torch.cuda.synchronize()
    seen.clear()
    before = {k: v.clone() for k, v in m.ada_state.items()}
    tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=2)
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(m.ada_state[k], v), "enable_cuda_graphs moved ada_state[%r]" % k
    captured = seen[-1]       # the captured D step's logits: static buffers the replays overwrite
    records, ps = [], []
    for _ in range(12):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        records.append(m.ada_state["record"].cpu().numpy().copy())
        _check_record(records[-1], captured, batch["label"].shape[0])
        ps.append(float(m.ada_state["p"]))
    acc0, pos0, p0 = before["acc"].cpu().numpy(), int(before["pos"]), float(before["p"])
    acc, pos, p, want = acc0.copy(), pos0, p0, []
    for rec in records:
        acc, pos, p = np_ada(acc, pos, p, rec, 0.6, 0.1, 2)
        want.append(p)
    assert ps == want and len(set(ps)) > 1, ps
    assert m.ada_state["acc"].cpu().numpy().tobytes() == acc.tobytes()
    tr.disable_cuda_graphs()


# ------------------------------------------------------------------------------------------ call trace
def test_call_trace_default_p_is_todays_and_ada_adds_exactly_the_new_calls(tmp_path):
    torch.cuda.set_device(0)
    policy = "color,translation,cutout"
    tr_off, _, batch = _trainer(str(tmp_path), "")
    tr_da, _, _ = _trainer(str(tmp_path), policy)
    tr_p1, _, _ = _trainer(str(tmp_path), policy, diff_augment_p=1.0)
    tr_ada, _, _ = _trainer(str(tmp_path), policy, ada_target=0.6)
    assert tr_da.pix2pix_model.ada_state is None and tr_p1.pix2pix_model.ada_state is None
    n_d = 2
    for _ in range(2):
        off, _ = _traced_step(tr_off, batch)
        da, n_da = _traced_step(tr_da, batch)
        p1, n_p1 = _traced_step(tr_p1, batch)
        ada, n_ada = _traced_step(tr_ada, batch)
        today = []       # tests/test_gpu_diffaug.py: the --diff_augment trace derived from the default one
        for c in off:
            if c == "s2e_make_d_input":
                today += ["s2e_diffaug_draw", "s2e_diffaug_means", "s2e_make_d_input_aug"]
            elif c == "s2e_d_input_grad":
                today.append("s2e_d_input_grad_aug")
            else:
                today.append(c)
        assert da == today and p1 == today and n_p1 == n_da
        # ADA: the gated twins, the D step's logit heads with the sign slot, and one controller launch before D's Adam
        want = [{"s2e_diffaug_draw": "s2e_diffaug_draw_p", "s2e_make_d_input_aug": "s2e_make_d_input_aug_masked",
                 "s2e_d_input_grad_aug": "s2e_d_input_grad_aug_masked"}.get(c, c) for c in today]
        d_start = len(want) - 1 - want[::-1].index("s2e_diffaug_draw_p")
        heads = [i for i in range(d_start, len(want)) if want[i] == "s2e_head_gather"]
        assert len(heads) == n_d
        for i in heads:
            want[i] = "s2e_head_gather_signs"
        want.insert(len(want) - 1 - want[::-1].index("s2e_adam_prepare"), "s2e_ada_update")
        assert ada == want
        # + the controller launch (the records' small torch copies and fills are not C-ABI calls)
        assert n_ada == n_da + 1


# ------------------------------------------------------------------------------------------ two ranks
def _worker(rank, world, port, tmp, q, backend):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                          LOCAL_RANK=str(rank))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        import torch.distributed as dist
        kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
        dist.init_process_group(backend, timeout=datetime.timedelta(seconds=90), rank=rank, world_size=world, **kw)
        from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
        oopt, opt = _opts(tmp, "color,translation,cutout", **ADA)
        opt.gpu_ids = [dev]
        torch.manual_seed(100 + rank)
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        m = tr.pix2pix_model
        _load(m, _sds(oopt, 81))
        full = O.synth_batch(oopt, 2 * world, 84)
        shard = {k: v[2 * rank:2 * rank + 2].clone() for k, v in full.items()}
        own, summed, ps = [], [], []
        real_allreduce = dist.all_reduce

        def spy(t, *a, **k):
            if t is m.ada_state["record"]:
                own.append(t.cpu().clone())
                out = real_allreduce(t, *a, **k)
                summed.append(t.cpu().clone())
                return out
            return real_allreduce(t, *a, **k)
        dist.all_reduce = spy
        use_graphs = backend == "nccl"
        for it in range(6):
            if use_graphs and it == 2:
                dist.all_reduce = real_allreduce
                tr.enable_cuda_graphs({k: v.cuda() for k, v in shard.items()}, warmup=2)
            d = {k: v.clone() for k, v in shard.items()}
            tr.run_generator_one_step(d)
            tr.run_discriminator_one_step(d)
            torch.cuda.synchronize()
            ps.append(m.ada_state["p"].cpu().numpy().copy())
        dist.all_reduce = real_allreduce
        own_all = [None] * world
        dist.all_gather_object(own_all, [o.numpy() for o in own])
        q.put((rank, dict(ps=np.stack(ps), summed=[s.numpy() for s in summed], own_all=own_all), None))
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
    res = {rank: r for rank, r, _ in got}
    r0 = res[0]
    for r in res.values():      # bitwise the same p on every rank after every D step
        assert r["ps"].tobytes() == r0["ps"].tobytes()
    assert len(set(r0["ps"].ravel().tolist())) > 1      # p moved
    own = r0["own_all"]
    for step, s in enumerate(r0["summed"]):      # the all-reduced record is the sum of the ranks' own records
        assert np.array_equal(s, sum(own[k][step] for k in range(world))), step
        assert s[-1] == 2 * world
    return r0


def test_two_ranks_on_one_gpu_keep_one_p(tmp_path):
    """gloo, both ranks on GPU 0, eager."""
    r0 = _run(str(tmp_path), "gloo")
    assert len(r0["summed"]) == 6


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpus_keep_one_p_with_graphs(tmp_path):
    """NCCL, one GPU per rank, CUDA graphs after two eager steps (the record's all-reduce between the two graphs)."""
    _run(str(tmp_path), "nccl")
