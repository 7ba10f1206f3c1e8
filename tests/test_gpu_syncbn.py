"""Synchronised SPADE BatchNorm (`--norm_G spectralspadesyncbatch3x3`) on real GPUs.

  * kernels, ranks simulated by batch shards on one GPU: s2e_norm_merge of per-shard s2e_norm_stats records equals the
    statistics of the whole batch (channels 200 sigma from zero, shards whose means differ by several sigma, an empty
    shard, up-sampled sources); s2e_spade_style_bwd_reduce per shard + summed sums + s2e_spade_style_bwd_apply per shard
    equals s2e_spade_style_bwd on the whole batch;
  * world size 1: `syncbatch` runs exactly the kernels of `batch` and computes the same values, eager and CUDA graphs;
  * two ranks (gloo, both on GPU 0): shards of 2 with shared statistics == one model on the batch of 4; running buffers
    bitwise equal on both ranks; the number of collectives per step;
  * two ranks on two GPUs (NCCL; skipped with fewer): the same, plus CUDA-graph replay == eager."""
import datetime
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.multiprocessing as mp

from oracle import seg2eye_oracle as O

pytestmark = pytest.mark.gpu
F64 = torch.float64
TOL_ACT = 1e-2      # tests/test_gpu_kernels.py test_spade_style_fwd_bwd


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


@pytest.fixture(scope="module")
def S():
    from seg2eye_b200 import _lib as L, ops
    L.lib()
    return L, ops


# ------------------------------------------------------------------------------------------ kernels, simulated ranks
SPLITS = {2: [3, 8], 3: [5, 0, 6], 8: [1, 2, 0, 3, 1, 1, 2, 1]}


def _record(L, x):
    B, H, W, C = x.shape
    rec = torch.empty(3 * C + 1, dtype=F64, device="cuda")
    L.call("s2e_norm_stats", L.ptr(x), B, H * W, C, 0, L.ptr(rec), L.stream())
    rec[3 * C] = B * H * W
    return rec


@pytest.mark.parametrize("up", [False, True])
@pytest.mark.parametrize("K", sorted(SPLITS))
def test_merged_statistics_equal_global_batch(S, K, up):
    L, ops = S
    sizes = SPLITS[K]
    g = torch.Generator().manual_seed(30 + K)
    B, H, W, C = sum(sizes), 24, 20, 64
    sigma = 0.25
    x = torch.randn(B, H, W, C, generator=g) * sigma + 50.0 * (1 + torch.arange(C).float() / C)     # 200 sigma from zero
    off = torch.repeat_interleave(torch.arange(K).float() * 6 * sigma, torch.tensor(sizes))       # shard means 6 sigma apart
    x = (x + off.view(B, 1, 1, 1)).to(torch.bfloat16).cuda()
    shards = torch.split(x, sizes)
    recs = torch.stack([_record(L, s) for s in shards]).reshape(-1)
    acc = torch.empty(3 * C, dtype=F64, device="cuda")
    cnt = torch.empty(1, dtype=F64, device="cuda")
    L.call("s2e_norm_merge", L.ptr(recs), K, C, L.ptr(acc), L.ptr(cnt), L.stream())
    mean, rstd = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    rm0, rv0 = torch.randn(C) * 0.1, torch.rand(C) + 0.5
    rm, rv, nbt = rm0.cuda(), rv0.cuda(), torch.tensor(5, device="cuda")
    fac = 4.0 if up else 1.0
    L.call("s2e_norm_finalize_merged", L.ptr(acc), L.ptr(cnt), C, fac, 1e-5, L.ptr(mean), L.ptr(rstd), L.ptr(rm), L.ptr(rv),
           0.1, L.ptr(nbt), L.stream())
    torch.cuda.synchronize()
    xd = x.double().cpu()
    n = B * H * W
    m_ref = xd.mean(dim=(0, 1, 2))
    v_ref = xd.var(dim=(0, 1, 2), unbiased=False)
    r_ref = 1.0 / torch.sqrt(v_ref + 1e-5)
    assert float(cnt) == n
    assert float(((mean.double().cpu() - m_ref).abs() / m_ref.abs()).max()) < 1e-6
    assert float(((rstd.double().cpu() - r_ref).abs() / r_ref).max()) < 1e-4
    cu = n * fac        # up: the normalised tensor has 4x the elements the statistics were summed over
    assert torch.allclose(rm.double().cpu(), 0.9 * rm0.double() + 0.1 * m_ref, rtol=1e-6, atol=1e-6)
    assert torch.allclose(rv.double().cpu(), 0.9 * rv0.double() + 0.1 * v_ref * cu / (cu - 1), rtol=1e-5, atol=1e-6)
    assert int(nbt) == 6
    # a rank that normalised with its own shard's statistics would be far off on this input (the test can fail)
    s0 = shards[0]
    a0 = torch.empty(3 * C, dtype=F64, device="cuda")
    L.call("s2e_norm_stats", L.ptr(s0), s0.shape[0], H * W, C, 0, L.ptr(a0), L.stream())
    m0, r0 = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    L.call("s2e_norm_finalize", L.ptr(a0), 1, C, float(s0.numel() // C), 0.0, 1e-5, L.ptr(m0), L.ptr(r0), None, None, 0.1,
           None, L.stream())
    assert float(((r0.double().cpu() - r_ref).abs() / r_ref).max()) > 100 * 1e-4
    assert float(((m0.double().cpu() - m_ref).abs() / m_ref.abs()).max()) > 100 * 1e-6


def _bwd_full(L, dout, amask, x, gb, style, mean, rstd, act, up_w):
    B, Hs, Ws, C = x.shape
    HW = dout.shape[1] * dout.shape[2]
    racc = torch.empty(B * 6 * C + 2 * C + 1, dtype=F64, device="cuda")
    dx, dgb = torch.empty_like(x), torch.empty_like(gb)
    dstyle = torch.empty_like(style) if style is not None else None
    chsum = torch.empty(3 * C, device="cuda")
    L.call("s2e_spade_style_bwd", L.ptr(dout), L.ptr(amask), L.ptr(x), L.ptr(gb), L.ptr(style), L.ptr(mean), L.ptr(rstd), B, HW,
           C, 0, act, L.ptr(racc), L.ptr(dx), 0, L.ptr(dgb), L.ptr(dstyle), L.ptr(chsum), up_w, 0, L.stream())
    return dx, dgb, dstyle, chsum


@pytest.mark.parametrize("plain", [False, True])
@pytest.mark.parametrize("up", [False, True])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_split_backward_with_summed_sums_equals_global_batch(S, act, up, plain):
    L, ops = S
    g = torch.Generator().manual_seed(40 + act + 3 * up)
    sizes = [2, 0, 3]
    B, H, W, C = sum(sizes), 12, 10, 64
    Hs, Ws = (H // 2, W // 2) if up else (H, W)
    x = (torch.randn(B, Hs, Ws, C, generator=g) * 1.5 + 0.3).to(torch.bfloat16).cuda()
    gb = (torch.randn(B, H, W, 2 * C, generator=g) * 0.5).to(torch.bfloat16).cuda()
    style = None if plain else (torch.randn(B, 2 * C, generator=g) * 0.5).cuda()
    dout = torch.randn(B, H, W, C, generator=g).to(torch.bfloat16).cuda()
    st = L.stream()
    acc = torch.empty(3 * C, dtype=F64, device="cuda")
    L.call("s2e_norm_stats", L.ptr(x), B, Hs * Ws, C, 0, L.ptr(acc), st)
    mean, rstd = torch.empty(1, C, device="cuda"), torch.empty(1, C, device="cuda")
    L.call("s2e_norm_finalize", L.ptr(acc), 1, C, float(B * Hs * Ws), float(B * H * W), 1e-5, L.ptr(mean), L.ptr(rstd), None,
           None, 0.1, None, st)
    out = torch.empty(B, H, W, C, dtype=torch.bfloat16, device="cuda")
    amask = torch.empty(B * H * W * (C // 8), dtype=torch.uint8, device="cuda") if act else None
    up_w = W if up else 0
    L.call("s2e_spade_style_fwd", L.ptr(x), L.ptr(gb), L.ptr(style), L.ptr(mean), L.ptr(rstd), B, H * W, C, 0, act, L.ptr(out),
           L.ptr(amask), up_w, st)
    dx_f, dgb_f, dst_f, _ = _bwd_full(L, dout, amask, x, gb, style, mean, rstd, act, up_w)

    bounds = [sum(sizes[:i]) for i in range(len(sizes) + 1)]
    mpp = H * W * (C // 8)      # mask bytes per sample
    parts, sums = [], []
    for b0, b1 in zip(bounds[:-1], bounds[1:]):
        n = b1 - b0
        p = dict(dout=dout[b0:b1], amask=amask[b0 * mpp:b1 * mpp] if act else None, x=x[b0:b1], gb=gb[b0:b1],
                 style=style[b0:b1] if style is not None else None)
        p["racc"] = torch.empty(n * 6 * C + 1, dtype=F64, device="cuda")
        p["dstyle"] = torch.empty_like(p["style"]) if style is not None else None
        s = torch.full((2 * C + 1,), float("nan"), dtype=F64, device="cuda")
        L.call("s2e_spade_style_bwd_reduce", L.ptr(p["dout"]), L.ptr(p["amask"]), L.ptr(p["x"]), L.ptr(p["gb"]), L.ptr(p["style"]),
               L.ptr(mean), L.ptr(rstd), n, H * W, C, 0, act, L.ptr(p["racc"]), L.ptr(s), L.ptr(p["dstyle"]), None, up_w, 0, st)
        parts.append(p)
        sums.append(s)
    total = torch.stack(sums).sum(0)       # what the all-reduce of the ranks' sums computes
    assert float(total[2 * C]) == B * H * W
    worst = 0.0
    for (b0, b1), p in zip(zip(bounds[:-1], bounds[1:]), parts):
        n = b1 - b0
        dx, dgb = torch.empty_like(p["x"]), torch.empty_like(p["gb"])
        L.call("s2e_spade_style_bwd_apply", L.ptr(p["dout"]), L.ptr(p["amask"]), L.ptr(p["x"]), L.ptr(p["gb"]), L.ptr(p["style"]),
               L.ptr(mean), L.ptr(rstd), n, H * W, C, 0, act, L.ptr(p["racc"]), L.ptr(total), L.ptr(dx), 0, L.ptr(dgb), up_w, 0, st)
        if n == 0:
            continue
        errs = [rel(dx, dx_f[b0:b1]), rel(dgb[..., :C], dgb_f[b0:b1, ..., :C]), rel(dgb[..., C:], dgb_f[b0:b1, ..., C:])]
        if style is not None:
            errs.append(rel(p["dstyle"], dst_f[b0:b1]))
        assert max(errs) < TOL_ACT, errs
        worst = max(worst, errs[0])
    # the shard's own sums alone give a different gradient (the test can fail)
    p = parts[0]
    dx0, dgb0 = torch.empty_like(p["x"]), torch.empty_like(p["gb"])
    L.call("s2e_spade_style_bwd_apply", L.ptr(p["dout"]), L.ptr(p["amask"]), L.ptr(p["x"]), L.ptr(p["gb"]), L.ptr(p["style"]),
           L.ptr(mean), L.ptr(rstd), sizes[0], H * W, C, 0, act, L.ptr(p["racc"]), L.ptr(sums[0]), L.ptr(dx0), 0, L.ptr(dgb0), up_w,
           0, st)
    assert rel(dx0, dx_f[:sizes[0]]) > max(10 * worst, 2e-3), (rel(dx0, dx_f[:sizes[0]]), worst)


# ------------------------------------------------------------------------------------------ world size 1
def _opts(tmp, norm_G, ngf, **kw):
    o = O.make_opt(ngf=ngf, ndf=16, lambda_l1=10.0, norm_G=norm_G, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[0], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=tmp, name="sbn", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale")
    return o, SimpleNamespace(**d)


def _one_iteration(tmp, norm_G, ngf, graphs, sds, batch):
    """One seeded G + D iteration at world size 1: C-ABI calls in order, and what the G step computes before its optimizer
    step (losses, image, G/E gradients, SPADE buffers)."""
    import contextlib
    import io
    from seg2eye_b200 import _lib as L
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    oopt, opt = _opts(tmp, norm_G, ngf)
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    m = tr.pix2pix_model
    nets = ((m.netG, "G"), (m.netD, "D"), (m.netE, "E"))
    for net, k in nets:
        net.load_state_dict({a: b.clone() for a, b in sds[k].items()})
    calls = []
    real = L.call

    def rec(name, *args):
        calls.append(name)
        return real(name, *args)
    L.call = rec     # the capture (graph mode) or the eager iteration: every C-ABI call in order
    try:
        if graphs:
            tr.enable_cuda_graphs({k: v.cuda() for k, v in batch.items()}, warmup=1)
        d = {k: v.clone() for k, v in batch.items()}
        tr.run_generator_one_step(d)
        gen = tr.get_latest_generated().detach().clone()
        g_grads = {"G." + n: p.grad.detach().clone() for n, p in m.netG.named_parameters() if p.grad is not None}
        g_grads.update({"E." + n: p.grad.detach().clone() for n, p in m.netE.named_parameters() if p.grad is not None})
        g_grads.update({"buf." + n: b.detach().clone() for n, b in m.netG.named_buffers() if "running" in n})
        g_grads.update({"loss." + k: v.detach().clone().reshape(-1) for k, v in tr.g_losses.items()})
        tr.run_discriminator_one_step(d)
        torch.cuda.synchronize()
    finally:
        L.call = real
    out = {"generated": gen}
    out.update(g_grads)
    if graphs:
        tr.disable_cuda_graphs()
    return out, calls


@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("ngf", [16, 64])
def test_world_size_one_syncbatch_is_batch(tmp_path, ngf, graphs):
    """`syncbatch` with one process runs the C-ABI calls of `batch`, in the same order, and computes the same G step.  The
    step itself reproduces to rounding only (float atomics in the weight-gradient, loss and statistics reductions), so
    the values are compared against that spread, measured by a second run of `batch`."""
    torch.cuda.set_device(0)
    oopt, _ = _opts(str(tmp_path), "spectralspadebatch3x3", ngf)
    sds = dict(G=O.synth_state(O.generator_shapes(oopt), 81), D=O.synth_state(O.discriminator_shapes(oopt), 82),
               E=O.synth_state(O.encoder_shapes(oopt), 83))
    batch = O.synth_batch(oopt, 2, 84)
    a, calls_a = _one_iteration(str(tmp_path), "spectralspadebatch3x3", ngf, graphs, sds, batch)
    a2, _ = _one_iteration(str(tmp_path), "spectralspadebatch3x3", ngf, graphs, sds, batch)
    s, calls_s = _one_iteration(str(tmp_path), "spectralspadesyncbatch3x3", ngf, graphs, sds, batch)
    assert calls_s == calls_a
    assert set(s) == set(a) and any(k.startswith("buf.") for k in a)
    spread = max(rel(a2[k], a[k]) for k in a)
    worst = max((rel(s[k], a[k]), k) for k in a)
    print("ngf %d graphs %d: syncbatch vs batch %.2e (%s), batch vs batch %.2e" % (ngf, graphs, worst[0], worst[1], spread))
    assert worst[0] <= max(4 * spread, 1e-3), (worst, spread)


# ------------------------------------------------------------------------------------------ two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, tmp, q, backend, norm_G, graphs):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                          LOCAL_RANK=str(rank))
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        import torch.distributed as dist
        # a short collective timeout: a desynchronised rank must fail the test, not hang the box
        kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
        dist.init_process_group(backend, timeout=datetime.timedelta(seconds=90), rank=rank, world_size=world, **kw)
        from seg2eye_b200 import ops
        from seg2eye_b200.models.pix2pix_model import Pix2PixModel
        from seg2eye_b200.models.networks.normalization import SPADE
        from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
        oopt, opt = _opts(tmp, norm_G, 16)
        opt.gpu_ids = [dev]
        torch.manual_seed(100 + rank)
        tr = Pix2PixTrainer(opt)
        m = tr.pix2pix_model
        sds = dict(G=O.synth_state(O.generator_shapes(oopt), 71), D=O.synth_state(O.discriminator_shapes(oopt), 72),
                   E=O.synth_state(O.encoder_shapes(oopt), 73))
        full = O.synth_batch(oopt, 2 * world, 74)
        shard = {k: v[2 * rank:2 * rank + 2].clone() for k, v in full.items()}
        names = ["fc.weight", "head_0.conv_0.weight_orig", "up_1.norm_0.spade.mlp_gamma.weight", "up_3.conv_1.weight_orig",
                 "up_3.norm_1.adain.linear.weight", "conv_img.weight", "head_0.norm_0.spade.mlp_shared.0.weight",
                 "up_0.norm_s.spade.mlp_beta.bias"]
        pG = dict(m.netG.named_parameters())
        res = {}

        def reload():
            for net, k in ((m.netG, "G"), (m.netD, "D"), (m.netE, "E")):
                net.load_state_dict({a: b.clone() for a, b in sds[k].items()})
            for o_ in (tr.optimizer_G, tr.optimizer_D):
                o_.state.clear()
                for g in o_.param_groups:
                    g.pop('_s2e_state', None)

        def two_iterations():
            out = []
            for _ in range(2):
                d = {k: v.clone() for k, v in shard.items()}
                tr.run_generator_one_step(d)
                tr.run_discriminator_one_step(d)
                out.append(torch.stack([v.reshape(-1)[0].detach().float() for v in tr.get_latest_losses().values()]).cpu())
            return out

        reload()
        m.train()
        if graphs:   # multi-rank CUDA graphs (shared statistics captured inside the [fwd+bwd] graphs) == multi-rank eager
            tr.enable_cuda_graphs({k: v.cuda() for k, v in shard.items()}, warmup=1)
            graph = two_iterations()
            tr.disable_cuda_graphs()
            reload()
            eager = two_iterations()
            res["graph_vs_eager"] = [float((a - b).abs().max()) for a, b in zip(eager, graph)]
            res["eager_losses"] = eager[1]
            tr.g_losses = tr.d_losses = None
            tr.generated = None
            reload()
        spades = [(n, mod) for n, mod in m.netG.named_modules() if isinstance(mod, SPADE)]
        # (1) rank 0 alone: a `spectralspadebatch3x3` model with the same weights on the WHOLE batch
        if rank == 0:
            _, opt_b = _opts(tmp, "spectralspadebatch3x3", 16)
            opt_b.gpu_ids = [dev]
            mb = Pix2PixModel(opt_b)
            for net, k in ((mb.netG, "G"), (mb.netD, "D"), (mb.netE, "E")):
                net.load_state_dict({a: b.clone() for a, b in sds[k].items()})
            mb.train()
            losses_f, _ = mb({k: v.clone() for k, v in full.items()}, mode='generator')
            sum(losses_f.values()).mean().backward()
            pB = dict(mb.netG.named_parameters())
            g_full = {n: pB[n].grad.detach().clone() for n in names}
            res["losses_full"] = torch.stack([v.reshape(-1)[0].detach() for v in losses_f.values()]).cpu()
            bufs_full = {n: (mod.param_free_norm.running_mean.clone(), mod.param_free_norm.running_var.clone())
                         for n, mod in dict(mb.netG.named_modules()).items() if isinstance(mod, SPADE)}
            del losses_f, mb
        tr.reducer_G.remove_hooks()
        dist.barrier()
        # (2) both ranks: sharded G step, gradients summed across ranks, collectives counted
        tr.optimizer_G.zero_grad()
        tr.reducer_G.armed, tr.reducer_D.armed = True, False
        n0 = ops._state.get("sync_collectives", 0)
        losses, _ = tr._fb('G', dict(shard))
        res["collectives_G"] = ops._state.get("sync_collectives", 0) - n0
        tr.reducer_G.allreduce()
        lsum = torch.stack([v.reshape(-1)[0].detach() for v in losses.values()])
        dist.all_reduce(lsum)
        res["losses_sharded_mean"] = (lsum / world).cpu()
        del losses
        bufs = {n: (mod.param_free_norm.running_mean.clone(), mod.param_free_norm.running_var.clone()) for n, mod in spades}
        flat = torch.cat([torch.cat(v) for v in bufs.values()])
        every = torch.empty(world * flat.numel(), dtype=flat.dtype, device=flat.device)
        dist.all_gather_into_tensor(every, flat)
        res["buffers_bitwise_equal"] = bool(torch.equal(every[:flat.numel()], every[flat.numel():]))
        if rank == 0:
            res["grad_err"] = {n: rel(pG[n].grad, g_full[n]) for n in names}
            res["rv_err"] = {n: rel(bufs[n][1], bufs_full[n][1]) for n in bufs}
            res["rm_err"] = {n: float((bufs[n][0] - bufs_full[n][0]).abs().max() / bufs_full[n][1].sqrt().norm()) for n in bufs}
        # (3) the D step's generator pass (no autograd graph): one collective per distinct SPADE input
        tr.reducer_G.armed, tr.reducer_D.armed = False, True
        n0 = ops._state.get("sync_collectives", 0)
        tr.optimizer_D.zero_grad()
        tr._fb('D', dict(shard))
        res["collectives_D"] = ops._state.get("sync_collectives", 0) - n0
        torch.cuda.synchronize()
        q.put((rank, res, None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:      # noqa: BLE001 -- report to the parent instead of hanging it
        import traceback
        q.put((rank, None, traceback.format_exc()))


def _run(tmp, backend, norm_G, graphs, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, tmp, q, backend, norm_G, graphs), daemon=True)
             for r in range(world)]
    for p in procs:
        p.start()
    got = []
    try:
        for _ in procs:
            got.append(q.get(timeout=400))
            if got[-1][2] is not None:      # a rank failed: its peers are stuck in a collective, do not wait for them
                break
    finally:
        for p in procs:
            p.join(5 if (got and got[-1][2] is not None) else 60)
            if p.is_alive():
                p.kill()
    for rank, res, err in got:
        assert err is None, "rank %d: %s" % (rank, err)
    assert len(got) == world
    return {rank: r for rank, r, _ in got}


def _check(res, sync):
    r0 = res[0]
    print("%s: grad_err %s\nlosses sharded %s full %s\nrv_err max %.3e rm_err max %.3e buffers equal on ranks %s collectives G %d D %d" % (
        "syncbatch" if sync else "batch", r0["grad_err"], r0["losses_sharded_mean"].tolist(), r0["losses_full"].tolist(),
        max(r0["rv_err"].values()), max(r0["rm_err"].values()), r0["buffers_bitwise_equal"], r0["collectives_G"], r0["collectives_D"]))
    if not sync:
        # per-rank statistics: the ranks' buffers drift apart, no collectives
        assert not r0["buffers_bitwise_equal"] and r0["collectives_G"] == 0 and r0["collectives_D"] == 0
        return
    vals = sorted(r0["grad_err"].values())
    assert vals[len(vals) // 2] < 5e-2 and vals[-1] < 1e-1, r0["grad_err"]
    assert torch.allclose(r0["losses_sharded_mean"], r0["losses_full"], rtol=2e-2, atol=2e-2)
    assert all(r["buffers_bitwise_equal"] for r in res.values())
    assert max(r0["rv_err"].values()) < 2e-2, r0["rv_err"]
    assert max(r0["rm_err"].values()) < 2e-2, r0["rm_err"]
    # 18 SPADE layers: 14 distinct inputs (norm_0 / norm_s of the 4 blocks with a learned shortcut share theirs) -> 14
    # all-gathers forward, 18 all-reduces backward; the D step's generator pass gathers its 14 again
    assert r0["collectives_G"] == 14 + 18 and r0["collectives_D"] == 14, (r0["collectives_G"], r0["collectives_D"])
    if "graph_vs_eager" in r0:
        assert r0["graph_vs_eager"][0] <= 2e-2 * float(r0["eager_losses"].abs().max()) + 2e-2, r0["graph_vs_eager"]
        assert r0["graph_vs_eager"][1] <= 5e-2 * float(r0["eager_losses"].abs().max()) + 2e-2, r0["graph_vs_eager"]


@pytest.mark.parametrize("norm_G", ["spectralspadesyncbatch3x3", "spectralspadebatch3x3"])
def test_two_ranks_on_one_gpu_match_full_batch(tmp_path, norm_G):
    """gloo, both ranks on GPU 0, eager (gloo collectives cannot be captured): the arithmetic of shared statistics."""
    _check(_run(str(tmp_path), "gloo", norm_G, False), "sync" in norm_G)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("norm_G", ["spectralspadesyncbatch3x3", "spectralspadebatch3x3"])
def test_two_gpus_match_full_batch_and_graph_path(tmp_path, norm_G):
    _check(_run(str(tmp_path), "nccl", norm_G, True), "sync" in norm_G)
