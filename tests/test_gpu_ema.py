"""`--ema_decay` on the device: the EMA instantiation of the multi-tensor Adam kernel and the multi-tensor byte copy
against host references, the trainer's averages against a float64 recurrence (eager and CUDA graphs), the default-off
path, the packed bf16 copies of the EMA nets, and two data-parallel ranks."""
import contextlib
import ctypes as C
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


def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _ramp(beta, t):
    """beta_t in fp32, as the kernel forms it: min(beta, (1 + t) / (10 + t))."""
    return np.float32(min(np.float32(beta), np.float32(1 + t) / np.float32(10 + t)))


def _adam(ts, state, ema=None, beta=0.0, lr_b=(0.0, 0.9), wd=0.0):
    from seg2eye_b200 import _lib as L
    p, g, m, v = ts
    n = len(p)
    s = L.stream()
    L.call("s2e_adam_prepare", L.ptr(state), lr_b[0], lr_b[1], s)
    args = (n, _ptrs(p), _ptrs(g), _ptrs(m), _ptrs(v), (C.c_longlong * n)(*[t.numel() for t in p]), L.ptr(state),
            lr_b[0], lr_b[1], 1e-8, wd)
    if ema is None:
        L.call("s2e_adam_multi", *args, s)
    else:
        L.call("s2e_adam_multi_ema", *args, _ptrs(ema), beta, s)


def _tensors(sizes, seed, misalign=()):
    """p away from zero and e within a factor 1.3 of p (same sign), so that e - p is exact in fp32 (Sterbenz) and the
    kernel's fmaf rounds once."""
    gen = torch.Generator().manual_seed(seed)
    out = {k: [] for k in "pgmve"}
    for i, n in enumerate(sizes):
        sign = torch.where(torch.rand(n, generator=gen) < 0.5, -1.0, 1.0)
        p = sign * (0.5 + torch.rand(n, generator=gen))
        vals = dict(p=p, g=torch.randn(n, generator=gen) * 1e-2, m=torch.randn(n, generator=gen) * 1e-3,
                    v=torch.rand(n, generator=gen) * 1e-4, e=p * (1 + 0.3 * (2 * torch.rand(n, generator=gen) - 1)))
        for k, t in vals.items():
            if i in misalign:       # a 4-byte offset view: the scalar path
                buf = torch.empty(n + 1, device="cuda")
                buf[1:].copy_(t)
                out[k].append(buf[1:])
            else:
                out[k].append(t.cuda())
    return out


SIZES = [1, 3, 5, 7, 4095, 4096, 4097, 3 * 4096 + 5, 10 * 4096, 33333]


@pytest.mark.parametrize("case", ["sizes", "many", "misaligned"])
@pytest.mark.parametrize("beta", [0.9, 0.999])
def test_adam_multi_ema_matches_adam_multi_and_fp64(case, beta):
    torch.cuda.set_device(0)
    if case == "many":      # more than 48 tensors: several launches
        sizes = [int(s) for s in np.random.default_rng(3).integers(1, 9000, size=113)]
    else:
        sizes = SIZES
    mis = (2, 5, 7) if case == "misaligned" else ()
    a, b = _tensors(sizes, 11, mis), _tensors(sizes, 11, mis)     # same values, same alignment (same kernel path)
    e0 = [t.double().cpu() for t in a["e"]]
    for step in (0, 5, 999):        # t = 1, 6, 1000 after prepare
        sa = torch.tensor([float(step), 1e-3, 0, 0], device="cuda")
        sb = sa.clone()
        _adam([a[k] for k in "pgmv"], sa)
        _adam([b[k] for k in "pgmv"], sb, ema=b["e"], beta=beta)
        torch.cuda.synchronize()
        assert torch.equal(sa, sb)
        for k in "pmv":
            for x, y in zip(a[k], b[k]):
                assert torch.equal(x, y), (k, x.numel())
        bt = float(_ramp(beta, step + 1))
        for i, (p, e) in enumerate(zip(b["p"], b["e"])):
            ref = (bt * (e0[i] - p.double().cpu()) + p.double().cpu()).numpy()
            got = e.cpu().numpy()
            ulp = np.spacing(np.abs(ref.astype(np.float32)))
            assert np.all(np.abs(got.astype(np.float64) - ref) <= ulp), (i, sizes[i], step)
            e0[i] = e.double().cpu()
        for k in "pgmv":      # the next round starts from identical inputs again
            for x, y in zip(a[k], b[k]):
                x.copy_(y)


@pytest.mark.parametrize("beta", [0.9, 0.999])
def test_ema_ramp_and_zero_decay(beta):
    """g = m = v = 0 leaves p unchanged, so with p = 0 and e = 1 the new e is beta_t itself."""
    torch.cuda.set_device(0)
    for t in (1, 2, 10, 1000):
        p, g, m, v = (torch.zeros(4099, device="cuda") for _ in range(4))
        e = torch.ones(4099, device="cuda")
        st = torch.tensor([float(t - 1), 1e-3, 0, 0], device="cuda")
        _adam([[p], [g], [m], [v]], st, ema=[e], beta=beta)
        torch.cuda.synchronize()
        assert float(st[0]) == t
        assert torch.all(e == float(_ramp(beta, t))), (t, float(e[0]), float(_ramp(beta, t)))
    a = _tensors(SIZES, 12)
    _adam([a[k] for k in "pgmv"], torch.tensor([3.0, 1e-3, 0, 0], device="cuda"), ema=a["e"], beta=0.0)
    torch.cuda.synchronize()
    for p, e in zip(a["p"], a["e"]):
        assert torch.equal(p, e)


def test_copy_multi_is_bitwise():
    from seg2eye_b200 import _lib as L
    torch.cuda.set_device(0)
    gen = torch.Generator().manual_seed(5)
    src = [torch.randint(-2 ** 62, 2 ** 62, (), generator=gen, dtype=torch.int64),     # num_batches_tracked
           torch.randn(64, generator=gen), torch.randn(17, generator=gen).double(),
           torch.randint(0, 255, (16385 * 3 + 7,), generator=gen, dtype=torch.uint8), torch.randn(100000, generator=gen)]
    src += [torch.randn(int(n), generator=gen) for n in np.random.default_rng(1).integers(1, 3000, size=60)]
    src = [s.cuda() for s in src]
    raw = torch.randint(0, 255, (1001,), dtype=torch.uint8, device="cuda")
    src.append(raw[3:1000])           # unaligned rows: the byte path
    dst = [torch.full_like(s, 7) for s in src]
    odd = torch.zeros(1001, dtype=torch.uint8, device="cuda")
    dst[-1] = odd[1:998]
    n = len(src)
    L.call("s2e_copy_multi", n, _ptrs(dst), _ptrs(src), (C.c_longlong * n)(*[s.numel() * s.element_size() for s in src]),
           L.stream())
    torch.cuda.synchronize()
    for d, s in zip(dst, src):
        assert torch.equal(d, s), (s.dtype, s.numel())
    assert int(odd[0]) == 0 and int(odd[998:].sum()) == 0     # nothing outside the rows


# ------------------------------------------------------------------------------------------ trainer
def _opts(tmp, ema_decay, ngf=16, **kw):
    o = O.make_opt(ngf=ngf, ndf=16, lambda_l1=10.0, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[0], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=tmp, name="ema", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale",
             ema_decay=ema_decay)
    return o, SimpleNamespace(**d)


def _sds(oopt, seed):
    return dict(G=O.synth_state(O.generator_shapes(oopt), seed), D=O.synth_state(O.discriminator_shapes(oopt), seed + 1),
                E=O.synth_state(O.encoder_shapes(oopt), seed + 2))


def _trainer(tmp, ema_decay, seed=31, **kw):
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    oopt, opt = _opts(tmp, ema_decay, **kw)
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    m = tr.pix2pix_model
    for net, k in ((m.netG, "G"), (m.netD, "D"), (m.netE, "E")):
        net.load_state_dict({a: b.clone() for a, b in _sds(oopt, seed)[k].items()})
    return tr, oopt, O.synth_batch(oopt, 2, seed + 3)


def _live_ema(m):
    live = [t for n in (m.netG, m.netE) for t in n.parameters()]
    ema = [t for n in (m.netG_ema, m.netE_ema) for t in n.parameters()]
    bl = [t for n in (m.netG, m.netE) for t in n.buffers()]
    be = [t for n in (m.netG_ema, m.netE_ema) for t in n.buffers()]
    return live, ema, bl, be


@pytest.mark.parametrize("graphs", [False, True])
def test_trainer_ema_follows_fp64_recurrence(tmp_path, graphs):
    torch.cuda.set_device(0)
    beta = 0.9
    tr, _, batch = _trainer(str(tmp_path), beta)
    m = tr.pix2pix_model
    m.sync_ema()        # the averages restart from the weights just loaded
    live, ema, bl, be = _live_ema(m)
    assert all(torch.equal(a, b) for a, b in zip(live, ema))
    if graphs:
        before = [t.detach().clone() for t in ema + be]
        tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=1)
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(before, ema + be)), "enable_cuda_graphs changed the averages"
    ref = [t.detach().double().cpu() for t in live]
    for step in range(1, 6):
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        torch.cuda.synchronize()
        assert float(tr.optimizer_G.param_groups[0]["_s2e_state"][0]) == step
        bt = float(_ramp(beta, step))
        ref = [bt * (r - p.detach().double().cpu()) + p.detach().double().cpu() for r, p in zip(ref, live)]
        for a, b in zip(be, bl):
            assert torch.equal(a, b)
        tr.run_discriminator_one_step(d)
    torch.cuda.synchronize()
    worst = max(float((e.double().cpu() - r).abs().max() / r.abs().max().clamp_min(1e-30)) for e, r in zip(ema, ref))
    moved = max(float((e.double().cpu() - p.detach().double().cpu()).abs().max()) for e, p in zip(ema, live))
    print("graphs %d: EMA vs fp64 recurrence %.2e, |EMA - live| max %.2e" % (graphs, worst, moved))
    assert worst <= 1e-6 and moved > 0
    if graphs:
        tr.disable_cuda_graphs()


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


def test_default_off_runs_todays_calls(tmp_path):
    torch.cuda.set_device(0)
    tr_off, _, batch = _trainer(str(tmp_path), 0.0)
    tr_on, _, _ = _trainer(str(tmp_path), 0.5)
    assert tr_off.pix2pix_model.netG_ema is None and tr_off.pix2pix_model.netE_ema is None
    for _ in range(2):
        off, n_off = _traced_step(tr_off, batch)
        on, n_on = _traced_step(tr_on, batch)
        assert "s2e_adam_multi_ema" not in off and "s2e_copy_multi" not in off
        # EMA on: the G step's Adam call becomes the EMA one and one buffer copy follows it
        assert on.count("s2e_adam_multi_ema") == 1 and on.count("s2e_copy_multi") == 1
        i = on.index("s2e_copy_multi")
        assert on[:i] + on[i + 1:] == [("s2e_adam_multi_ema" if c == "s2e_adam_multi" and k == i - 1 else c)
                                       for k, c in enumerate(off)]
        assert n_on == n_off + 1


@pytest.mark.parametrize("graphs", [False, True])
def test_pack_jobs_unchanged_and_ema_forwards_use_fresh_weights(tmp_path, graphs):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    torch.cuda.set_device(0)
    jobs = []
    real = ops._run_pack_jobs

    def count(js):
        jobs.append(len(js))
        return real(js)

    def step_jobs(tr, batch):
        jobs.clear()
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)
        return sum(jobs)

    tr_off, oopt, batch = _trainer(str(tmp_path), 0.0)
    tr_on, _, _ = _trainer(str(tmp_path), 0.9)
    m = tr_on.pix2pix_model
    if graphs:
        for tr in (tr_off, tr_on):
            tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=1)
    ops._run_pack_jobs = count
    try:
        for tr in (tr_off, tr_on):
            step_jobs(tr, batch)        # first step: the packed copies are created (eager)
        base = step_jobs(tr_off, batch)
        assert (base > 0 or graphs) and step_jobs(tr_on, batch) == base
        m.eval()
        with torch.no_grad():
            m({k: v.clone() for k, v in batch.items()}, mode="inference")     # registers the EMA nets' copies
        m.train()
        for _ in range(2):
            assert step_jobs(tr_on, batch) == base
            assert step_jobs(tr_off, batch) == base
        # the EMA nets called directly after further steps (no model mode involved)
        m.eval()
        seg, style, _ = m.preprocess_input({k: v.clone() for k, v in batch.items()})
        with torch.no_grad():
            mu_got = m.netE_ema.forward_samples(style)[0].clone()
            w = m._aggregate_tensor(mu_got).clone()
            img_got = m.netG_ema(seg, w).clone()
            # a second inference with no G step in between re-packs nothing
            m({k: v.clone() for k, v in batch.items()}, mode="inference")
            jobs.clear()
            m({k: v.clone() for k, v in batch.items()}, mode="inference")
            assert sum(jobs) == 0, jobs
    finally:
        ops._run_pack_jobs = real
    with torch.no_grad():
        got = m({k: v.clone() for k, v in batch.items()}, mode="inference").clone()
        w_got = m({k: v.clone() for k, v in batch.items()}, mode="encode_only").clone()
    # == a fresh model holding the averages
    _, opt_f = _opts(str(tmp_path), 0.0)
    with contextlib.redirect_stdout(io.StringIO()):
        fresh = Pix2PixModel(opt_f)
    fresh.netG.load_state_dict({k: v.clone() for k, v in m.netG_ema.state_dict().items()})
    fresh.netE.load_state_dict({k: v.clone() for k, v in m.netE_ema.state_dict().items()})
    fresh.eval()
    with torch.no_grad():
        want = fresh({k: v.clone() for k, v in batch.items()}, mode="inference")
        w_want = fresh({k: v.clone() for k, v in batch.items()}, mode="encode_only")
        mu_want = fresh.netE.forward_samples(style)[0]
        img_want = fresh.netG(seg, w)
        live = tr_on.pix2pix_model.netG.state_dict()
    rel = lambda a, b: float((a.float() - b.float()).norm() / b.float().norm())
    print("graphs %d: EMA vs fresh model: inference %.2e, encode_only %.2e, direct netE_ema %.2e, direct netG_ema %.2e"
          % (graphs, rel(got, want), rel(w_got, w_want), rel(mu_got, mu_want), rel(img_got, img_want)))
    assert rel(got, want) <= 1e-5 and rel(w_got, w_want) <= 1e-5
    assert rel(mu_got, mu_want) <= 1e-5 and rel(img_got, img_want) <= 1e-5
    assert any(not torch.equal(v, live[k]) for k, v in m.netG_ema.state_dict().items())
    if graphs:
        for tr in (tr_off, tr_on):
            tr.disable_cuda_graphs()


# ------------------------------------------------------------------------------------------ two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, tmp, q, backend, graphs):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                          LOCAL_RANK=str(rank))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        import torch.distributed as dist
        kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
        dist.init_process_group(backend, timeout=datetime.timedelta(seconds=90), rank=rank, world_size=world, **kw)
        from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
        # synchronised BatchNorm: the live buffers, hence their copies, are identical on every rank too
        oopt, opt = _opts(tmp, 0.9, norm_G="spectralspadesyncbatch3x3")
        opt.gpu_ids = [dev]
        torch.manual_seed(100 + rank)      # different initial weights per rank: the broadcast must align the averages
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        m = tr.pix2pix_model
        full = O.synth_batch(oopt, 2 * world, 74)
        shard = {k: v[2 * rank:2 * rank + 2].clone().cuda() for k, v in full.items()}
        _, ema, _, be = _live_ema(m)
        init = [t.detach().clone() for t in ema]
        if graphs:
            tr.enable_cuda_graphs(shard, warmup=1)
        for _ in range(3):
            d = dict(shard)
            tr.run_generator_one_step(d)
            tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
        flat = torch.cat([t.detach().reshape(-1).double() for t in ema + be])
        every = torch.empty(world * flat.numel(), dtype=flat.dtype, device=flat.device)
        dist.all_gather_into_tensor(every, flat)
        res = dict(equal=bool(torch.equal(every[:flat.numel()], every[flat.numel():])),
                   moved=any(not torch.equal(a, b) for a, b in zip(init, ema)))
        if graphs:
            tr.disable_cuda_graphs()
        q.put((rank, res, None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:      # noqa: BLE001 -- report to the parent instead of hanging it
        import traceback
        q.put((rank, None, traceback.format_exc()))


def _run(tmp, backend, graphs, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, tmp, q, backend, graphs), daemon=True) for r in range(world)]
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
    for _, res, _ in got:
        assert res["equal"] and res["moved"], res


def test_two_ranks_on_one_gpu_keep_identical_averages(tmp_path):
    """gloo, both ranks on GPU 0, eager: the average advances after the all-reduced step, identically on every rank."""
    _run(str(tmp_path), "gloo", False)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpus_keep_identical_averages_under_cuda_graphs(tmp_path):
    _run(str(tmp_path), "nccl", True)
