"""Module- and step-level parity on the GPU: the drop-in modules (seg2eye_b200.models.networks, Pix2PixModel,
Pix2PixTrainer) against the CPU oracle (itself pinned to the reference by tests/test_oracle_golden.py) and
against the committed reference outputs in tests/golden/ref_small.npz, on identical weights and inputs.

Tolerances (BASELINE.md section 5, bf16 inputs / fp32 accumulation):
  * module level (SURVEY 8(c)(ii): every SPADE_STYLE ResBlock / D level / E level given the oracle's input):
    forward activations <= 1e-2 relative L2 error (measured 3.5e-3 .. 4.4e-3 per ResBlock);
  * the chained 7-block generator accumulates those independent bf16 roundings: a CPU emulation that rounds the
    oracle at the same points (tools/precision_floor.py) predicts 1.1e-2 at up_3 and 1.8e-2 on the image for this small
    model, 1.4e-2 on the image from the bf16 OPERANDS alone; the device measures 1.2e-2 / 1.7-1.9e-2, so the end-to-end
    image bound against the oracle is TOL_CHAIN = 2.5e-2 (at the benchmarked width the image error is 1.1-1.4e-2,
    tests/test_gpu_fullsize.py); two noisy implementations compared with each other get TOL_PAIR = 3e-2;
  * G/D losses after one optimiser step <= 2e-2 relative (absolute floor 2e-2 for the hinge-G term, a mean of signed
    logits that nearly cancels)."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import seg2eye_oracle as O
from oracle.make_golden import IMAGE_SUB

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL_ACT = 1e-2
TOL_CHAIN = 2.5e-2
TOL_PAIR = 3e-2
TOL_LOSS = 2e-2


def rel(a, b):
    a = torch.as_tensor(np.asarray(a.detach().float().cpu() if torch.is_tensor(a) else a)).double()
    b = torch.as_tensor(np.asarray(b.detach().float().cpu() if torch.is_tensor(b) else b)).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def sub(t, n=4096):
    f = t.detach().float().cpu().reshape(-1).double()
    step = max(1, f.numel() // n)
    return f[::step][:n].float().numpy()


def make_opts(**kw):
    o = O.make_opt(**kw)
    d = vars(o).copy()
    d.update(gpu_ids=[0], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir="/tmp/s2e_ckpt", name="t", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale")
    return o, SimpleNamespace(**d)


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(GOLD, "ref_small.npz")))


@pytest.fixture(scope="module")
def ctx(gold):
    ngf, ndf, l1, bs = [int(x) for x in gold["meta_cfg"]]
    sG, sD, sE, sB = [int(x) for x in gold["meta_seeds"]]
    oopt, opt = make_opts(ngf=ngf, ndf=ndf, lambda_l1=float(l1))
    return SimpleNamespace(oopt=oopt, opt=opt, bs=bs, seeds=dict(G=sG, D=sD, E=sE, batch=sB),
                           batch=O.synth_batch(oopt, bs, sB))


def load(net, sd):
    net.load_state_dict({k: v.clone() for k, v in sd.items()})
    return net.cuda()


def test_encoder_forward(ctx, gold):
    from seg2eye_b200.models import networks
    sd = O.synth_state(O.encoder_shapes(ctx.oopt), ctx.seeds["E"])
    with torch.no_grad():
        mu_o, lv_o, feats_o = O.encoder_forward({k: v.clone() for k, v in sd.items()}, ctx.batch["style_image"][0], ctx.oopt)
    E = load(networks.ConvEncoder(ctx.opt), sd).train()
    with torch.no_grad():
        mu, lv, feats = E(ctx.batch["style_image"][0].cuda())
    for i, (a, b) in enumerate(zip(feats, feats_o)):
        assert rel(a, b) < TOL_ACT, (i, rel(a, b))
    assert rel(mu, mu_o) < TOL_ACT and rel(lv, lv_o) < TOL_ACT
    assert rel(mu, gold["E_mu"]) < TOL_ACT
    assert rel(E.state_dict()["layer0.0.weight_u"], gold["E_layer0_u_after"]) < 1e-4


def test_batched_encoder_equals_per_sample_calls(ctx):
    """ConvEncoder.forward_samples == the reference's loop of one netE call per sample (pix2pix_model.py:285):
    same mu, same advanced u/v buffers, same parameter gradients (incl. the spectral chain-rule term)."""
    from seg2eye_b200.models import networks
    sd = O.synth_state(O.encoder_shapes(ctx.oopt), ctx.seeds["E"])
    style = ctx.batch["style_image"].cuda()
    B = style.shape[0]
    g = torch.Generator().manual_seed(3)
    dmu = torch.randn(B, style.shape[1], 16, generator=g).cuda()
    res = {}
    for mode in ("loop", "batched"):
        E = load(networks.ConvEncoder(ctx.opt), sd).train()
        if mode == "loop":
            mu = torch.stack([E(style[b])[0] for b in range(B)], 0)
        else:
            mu = E.forward_samples(style)[0]
        (mu * dmu).sum().backward()
        res[mode] = (mu.detach(), {k: p.grad.clone() for k, p in E.named_parameters() if p.grad is not None},
                     {k: v.clone() for k, v in E.state_dict().items() if k.endswith("_u") or k.endswith("_v")})
    # the two paths round the conv outputs to bf16 at different scales (z vs z/sigma): one-ulp differences, amplified by
    # the 6-layer random-weight encoder like any other rounding noise (measured 9e-3) -> module-level bound
    assert rel(res["batched"][0], res["loop"][0]) < TOL_ACT
    for k, v in res["loop"][2].items():
        assert rel(res["batched"][2][k], v) < 1e-5, k            # u / v advanced B times, identically
    assert set(res["batched"][1]) == set(res["loop"][1])
    errs = {k: rel(res["batched"][1][k], v) for k, v in res["loop"][1].items()}
    assert max(errs.values()) < 0.1, errs
    # and against the CPU oracle's per-sample loop
    with torch.no_grad():
        w_o = O.encode_w({k: v.clone() for k, v in sd.items()}, ctx.batch["style_image"], ctx.oopt)
    assert rel(res["batched"][0].mean(1), w_o) < TOL_ACT


def test_generator_forward(ctx, gold):
    from seg2eye_b200.models import networks
    sd = O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"])
    seg = O.one_hot(ctx.batch["label"], 4)
    w = torch.from_numpy(gold["w"])
    sdo = {k: v.clone() for k, v in sd.items()}
    taps = {}
    with torch.no_grad():
        fake_o = O.generator_forward(sdo, seg, w, ctx.oopt, taps=taps)
    G = load(networks.SPADESTYLEGenerator(ctx.opt), sd).train()
    with torch.no_grad():
        fake = G(seg.cuda(), w.cuda())
    assert fake.shape == fake_o.shape and fake.dtype == torch.float32
    assert rel(fake, fake_o) < TOL_CHAIN, rel(fake, fake_o)
    assert rel(sub(fake, IMAGE_SUB), gold["G_fake_sub"]) < TOL_CHAIN
    post = G.state_dict()
    for k in ("head_0.norm_0.spade.param_free_norm.running_mean", "up_3.norm_1.spade.param_free_norm.running_var",
              "up_2.conv_0.weight_u", "up_2.conv_s.weight_v"):
        assert rel(post[k], sdo[k]) < TOL_ACT, k
        assert rel(post[k], gold["G_buf_" + k]) < TOL_ACT, k
    assert int(post["up_3.norm_1.spade.param_free_norm.num_batches_tracked"]) == int(
        gold["G_buf_up_3.norm_1.spade.param_free_norm.num_batches_tracked"])


def test_generator_blocks_match_oracle_taps(ctx):
    """Module-level parity: every SPADE_STYLE_ResnetBlock fed with the ORACLE's input must reproduce the oracle's
    output within 1e-2; the chained activations must stay within the accumulated-rounding bound."""
    from seg2eye_b200.models import networks
    from seg2eye_b200 import ops
    sd = O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"])
    seg = O.one_hot(ctx.batch["label"], 4)
    w = O.synth_state({"w": (ctx.bs, 16)}, 5, scale=4.0)["w"]
    taps = {}
    with torch.no_grad():
        O.generator_forward({k: v.clone() for k, v in sd.items()}, seg, w, ctx.oopt, taps=taps)
    G = load(networks.SPADESTYLEGenerator(ctx.opt), sd).train()
    G2 = load(networks.SPADESTYLEGenerator(ctx.opt), sd).train()
    G3 = load(networks.SPADESTYLEGenerator(ctx.opt), sd).train()
    segc, wc = seg.cuda(), w.cuda()
    nhwc = lambda t: t.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()
    with torch.no_grad():
        x = G.fc.forward_nhwc(ops.seg_nearest(segc, G.sh, G.sw))
        assert rel(x.permute(0, 3, 1, 2), taps["fc"]) < TOL_ACT
        chained, fed, fed_up, prev = {}, {}, {}, "fc"
        for name in ("head_0", "G_middle_0", "G_middle_1", "up_0", "up_1", "up_2", "up_3"):
            up = name != "head_0" and not (name == "G_middle_1" and ctx.opt.num_upsampling_layers == "normal")
            xin = taps[prev]
            if up:
                x = G.up(x)
                xin = xin.repeat_interleave(2, 2).repeat_interleave(2, 3)
            fed[name] = rel(getattr(G2, name).forward_nhwc(nhwc(xin), segc, wc).permute(0, 3, 1, 2), taps[name])
            if up:   # the same block fed with the LOW-resolution tensor: up-sampling folded into the SPADE kernels
                fed_up[name] = rel(getattr(G3, name).forward_nhwc(nhwc(taps[prev]), segc, wc, up=True).permute(0, 3, 1, 2), taps[name])
            x = getattr(G, name).forward_nhwc(x, segc, wc)
            chained[name] = rel(x.permute(0, 3, 1, 2), taps[name])
            prev = name
    assert max(fed.values()) < TOL_ACT, fed
    assert len(fed_up) == 5 and max(fed_up.values()) < TOL_ACT, fed_up
    # norm_s and norm_0 of the four blocks with a learned shortcut share one statistics pass over their common input
    assert ops._state.get("stats_shared", 0) >= 4, ops._state.get("stats_shared", 0)
    assert max(chained.values()) < TOL_CHAIN, chained


def test_discriminator_forward(ctx, gold):
    from seg2eye_b200.models import networks
    sd = O.synth_state(O.discriminator_shapes(ctx.oopt), ctx.seeds["D"])
    seg = O.one_hot(ctx.batch["label"], 4)
    # the reference's G_fake, recomputed by the oracle (pinned to its stored sample in tests/test_oracle_golden.py)
    with torch.no_grad():
        fake = O.generator_forward(O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"]), seg, torch.from_numpy(gold["w"]),
                                   ctx.oopt)
    both = torch.cat([torch.cat([seg, fake], 1), torch.cat([seg, ctx.batch["target"]], 1)], 0)
    with torch.no_grad():
        outs_o = O.discriminator_forward({k: v.clone() for k, v in sd.items()}, both, ctx.oopt)
    D = load(networks.MultiscaleDiscriminator(ctx.opt), sd).train()
    with torch.no_grad():
        outs = D(both.cuda())
    for i in range(2):
        for j in range(5):
            assert outs[i][j].shape == outs_o[i][j].shape
            assert rel(outs[i][j], outs_o[i][j]) < TOL_ACT, (i, j, rel(outs[i][j], outs_o[i][j]))
    assert rel(outs[0][4], gold["D_0_4"]) < TOL_ACT and rel(outs[1][4], gold["D_1_4"]) < TOL_ACT


def _loss_close(name, got, want):
    got, want = float(got), float(want)
    floor = 2e-2 if name == "GAN" else 0.0
    assert abs(got - want) <= TOL_LOSS * abs(want) + floor, (name, got, want)


def _make_trainer(ctx):
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    tr = Pix2PixTrainer(ctx.opt)
    m = tr.pix2pix_model
    load(m.netG, O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"]))
    load(m.netD, O.synth_state(O.discriminator_shapes(ctx.oopt), ctx.seeds["D"]))
    load(m.netE, O.synth_state(O.encoder_shapes(ctx.oopt), ctx.seeds["E"]))
    return tr


def test_two_training_iterations_vs_reference(ctx, gold):
    """Full G step + D step through Pix2PixTrainer, twice; losses of iteration 1 come after one optimiser step."""
    tr = _make_trainer(ctx)
    for it in range(2):
        data = {k: v.clone() for k, v in ctx.batch.items()}
        tr.run_generator_one_step(data)
        tr.run_discriminator_one_step(data)
        losses = tr.get_latest_losses()
        assert set(losses) == {"GAN", "L1/weighted", "GAN_Feat", "D/Fake", "D/real"}
        assert losses["GAN"].shape == (1,) and losses["GAN_Feat"].shape == (1,) and losses["D/real"].shape == (1,)
        for k, v in losses.items():
            _loss_close(k, v.reshape(-1)[0], gold["step%d_loss_%s" % (it, k)][0])
        # iteration 1 runs on weights moved by Adam(beta1=0) ~ lr*sign(g): every weight whose tiny gradient changes sign
        # under bf16 noise moves the other way, so the image bound after the step is loose (measured 4-5e-2); the
        # contractual quantities after the optimiser step are the losses (checked above at 2e-2)
        key = "G_fake" if it == 0 else "step%d_generated" % it     # iteration 0 generates G_fake again
        assert rel(sub(tr.get_latest_generated(), IMAGE_SUB), gold[key + "_sub"]) < (TOL_CHAIN if it == 0 else 1e-1)
    post = dict(G=tr.pix2pix_model.netG.state_dict(), D=tr.pix2pix_model.netD.state_dict(),
                E=tr.pix2pix_model.netE.state_dict())
    # parameters after two Adam(beta1=0) steps: each step moves every weight by ~lr*sign(g); compare the bulk
    for k, v in gold.items():
        if not k.startswith("post_") or k.endswith("_stat"):
            continue
        net, name = k[5], k[7:]
        if name.endswith("_sub"):
            assert rel(sub(post[net][name[:-4]]), v) < 2e-2, k
        elif name.endswith("num_batches_tracked"):
            assert int(post[net][name]) == int(v)
        else:
            assert rel(post[net][name], v) < 2e-2, k


def _grad_errors(ctx, **over):
    oopt = SimpleNamespace(**{**vars(ctx.oopt), **over})
    opt = SimpleNamespace(**{**vars(ctx.opt), **over})
    c2 = SimpleNamespace(oopt=oopt, opt=opt, bs=ctx.bs, seeds=ctx.seeds, batch=ctx.batch)
    tr = _make_trainer(c2)
    m = tr.pix2pix_model
    data = {k: v.clone() for k, v in ctx.batch.items()}
    m.train()
    from seg2eye_b200 import ops
    hits0 = ops._state.get("chsum_hits", 0)
    g_losses, _ = m(data, mode="generator")
    sum(g_losses.values()).mean().backward()
    # the SPADE+Style backward hands per-channel sums to the gamma|beta convs (18) and to every conv_0 (7): their bias
    # gradients must come from there, not from another pass over the gradient tensors
    assert ops._state.get("chsum_hits", 0) - hits0 >= 25, ops._state.get("chsum_hits", 0) - hits0
    gG = {k: p.grad.detach().cpu().clone() for k, p in m.netG.named_parameters() if p.grad is not None}
    gE = {k: p.grad.detach().cpu().clone() for k, p in m.netE.named_parameters() if p.grad is not None}
    assert all(p.grad is None for p in m.netD.parameters())   # D weight gradients are skipped in the G step
    sdG = O.synth_state(O.generator_shapes(oopt), ctx.seeds["G"])
    sdD = O.synth_state(O.discriminator_shapes(oopt), ctx.seeds["D"])
    sdE = O.synth_state(O.encoder_shapes(oopt), ctx.seeds["E"])
    O.OracleTrainer(sdG, sdD, sdE, oopt)
    losses_o, _ = O.generator_losses(sdG, sdD, sdE, ctx.batch, oopt)
    sum(losses_o.values()).mean().backward()
    errs = {"G." + k: rel(g, sdG[k].grad) for k, g in gG.items()}
    errs.update({"E." + k: rel(g, sdE[k].grad) for k, g in gE.items()})
    assert set(gG) == {k for k, v in sdG.items() if v.grad is not None}
    assert "fc_var.weight" not in gE  # never receives a gradient (encoder.py:71: logvar is unused)
    return errs


def test_gradients_match_oracle_smooth_losses(ctx):
    """G-step parameter gradients vs CPU autograd through the oracle with smooth losses only (hinge-G + L2).
    The LeakyReLU masks of D and G flip wherever a pre-activation is below the bf16 noise, which alone gives ~5 %
    (measured 5.6-5.9 %, uniform over all layers); the median over all G and E parameter gradients must be within 8e-2 relative L2, the worst within 0.5
    (per-(sample,channel) style gradients are sums with heavy cancellation)."""
    errs = _grad_errors(ctx, no_ganFeat_loss=True, lambda_l1=0.0, lambda_l2=10.0)
    vals = sorted(errs.values())
    worst = dict(sorted(((k, round(v, 3)) for k, v in errs.items()), key=lambda kv: -kv[1])[:6])
    assert vals[len(vals) // 2] < 8e-2, (vals[len(vals) // 2], worst)
    assert vals[-1] < 0.5, worst


def test_gradients_match_oracle_default_losses(ctx):
    """Same with the benchmark's losses (hinge + feature-matching L1 + image L1).  d|x|/dx = sign(x) flips wherever
    |fake - real| is below the bf16 activation noise, so the bound is looser: median <= 0.12, and <= 0.5 for the few
    gradients that are sums with heavy cancellation (per-(sample,channel) style gradients)."""
    errs = _grad_errors(ctx)
    vals = sorted(errs.values())
    assert vals[len(vals) // 2] < 0.12, vals[len(vals) // 2]
    bad = {k: round(v, 4) for k, v in errs.items() if v > 0.5}
    assert not bad, bad


def test_tcgen05_and_simt_paths_agree_on_a_step(ctx):
    from seg2eye_b200 import ops, _lib as L
    out = {}
    for impl in (L.IMPL_SIMT, None):
        tr = _make_trainer(ctx)
        data = {k: v.clone() for k, v in ctx.batch.items()}
        if impl is None:
            tr.run_generator_one_step(data)
        else:
            with ops.force_impl(impl):
                tr.run_generator_one_step(data)
        out[impl] = ({k: float(v.reshape(-1)[0]) for k, v in tr.g_losses.items()}, tr.generated.detach().cpu())
    # both paths round at the same points; accumulation-order differences (1-ulp flips, 1e-4 per conv) are amplified
    # by the random-weight network exactly like the bf16 drift itself (measured 2.0e-2 on the image)
    assert rel(out[None][1], out[L.IMPL_SIMT][1]) < TOL_PAIR
    for k in out[None][0]:
        assert abs(out[None][0][k] - out[L.IMPL_SIMT][0][k]) <= TOL_LOSS * abs(out[L.IMPL_SIMT][0][k]) + 2e-2, k


def test_cuda_graph_steps_match_eager(ctx):
    """enable_cuda_graphs() must be side-effect free and replayed iterations must equal eager iterations."""
    eager, graph = _make_trainer(ctx), _make_trainer(ctx)
    dev = {k: v.cuda() for k, v in ctx.batch.items()}
    before = {k: v.clone() for k, v in graph.pix2pix_model.netG.state_dict().items()}
    graph.enable_cuda_graphs(dev, warmup=2)
    after = graph.pix2pix_model.netG.state_dict()
    assert all(torch.equal(before[k], after[k]) for k in before), "graph capture changed the model state"
    for it in range(2):
        for tr in (eager, graph):
            data = {k: v.clone() for k, v in ctx.batch.items()}
            tr.run_generator_one_step(data)
            tr.run_discriminator_one_step(data)
        le, lg = eager.get_latest_losses(), graph.get_latest_losses()
        for k in le:
            a, b = float(le[k].reshape(-1)[0]), float(lg[k].reshape(-1)[0])
            # iteration 0, G losses: same kernels on the same data.  Everything later sees weights updated through
            # atomically-accumulated (order-dependent) weight gradients followed by Adam(beta1=0) ~ lr*sign(g)
            tight = it == 0 and not k.startswith("D/")
            assert abs(a - b) <= (2e-3 if tight else TOL_LOSS) * abs(a) + (1e-4 if tight else 2e-2), (it, k, a, b)
    assert rel(graph.get_latest_generated(), eager.get_latest_generated()) < TOL_PAIR
    nbt = "up_3.norm_0.spade.param_free_norm.num_batches_tracked"
    assert int(graph.pix2pix_model.netG.state_dict()[nbt]) == int(eager.pix2pix_model.netG.state_dict()[nbt])


def test_checkpoint_roundtrip_in_reference_layout(ctx, tmp_path):
    from seg2eye_b200 import util
    tr = _make_trainer(ctx)
    opt = SimpleNamespace(**{**vars(ctx.opt), "checkpoints_dir": str(tmp_path), "name": "ck"})
    tr.pix2pix_model.opt = opt
    tr.save("latest")
    for label, shapes in (("G", O.generator_shapes(ctx.oopt)), ("D", O.discriminator_shapes(ctx.oopt)),
                          ("E", O.encoder_shapes(ctx.oopt))):
        sd = torch.load(os.path.join(str(tmp_path), "ck", "latest_net_%s.pth" % label))
        assert list(sd.keys()) == list(shapes.keys())
        assert all(v.device.type == "cpu" for v in sd.values())
        assert all(v.dtype == (torch.int64 if k.endswith("num_batches_tracked") else torch.float32) for k, v in sd.items())
    util.load_network(tr.pix2pix_model.netG, "G", "latest", opt)


def test_inference_and_encode_only_modes(ctx, gold):
    """BASELINE config 4 path: mode='encode_only' -> w, interpolate, mode='inference' with `latent_style`
    (pix2pix_model.py:76-88).  Checked against the oracle's generator on the same w."""
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(ctx.opt)
    load(m.netG, O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"]))
    load(m.netE, O.synth_state(O.encoder_shapes(ctx.oopt), ctx.seeds["E"]))
    m.train()
    data = {k: v.clone() for k, v in ctx.batch.items()}
    w = m(data, mode="encode_only")
    assert w.shape == (ctx.bs, 16) and rel(w, gold["w"]) < TOL_ACT
    # interpolate between the two style codes, 3 steps, labels repeated
    alphas = torch.tensor([0.0, 0.5, 1.0], device=w.device).view(-1, 1)
    wi = (1 - alphas) * w[0:1] + alphas * w[1:2]
    lab = ctx.batch["label"][0:1].repeat(3, 1, 1, 1)
    out = m({"label": lab, "style_image": ctx.batch["style_image"][0:1].repeat(3, 1, 1, 1, 1), "latent_style": wi.detach()},
            mode="inference")
    assert out.shape == (3, 1, 320, 256) and out.dtype == torch.float32 and not out.requires_grad
    sdG = O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"])
    with torch.no_grad():
        ref = O.generator_forward(sdG, O.one_hot(lab, 4), wi.detach().cpu(), ctx.oopt)
    assert rel(out, ref) < TOL_CHAIN
    with pytest.raises(ValueError):
        m(data, mode="bogus")


@pytest.mark.parametrize("over", [dict(norm_G="spectralspadeinstance3x3"), dict(num_upsampling_layers="more", crop_size=512)])
def test_generator_variants_vs_oracle(ctx, over):
    """SPADE with InstanceNorm statistics (shard-invariant config of SURVEY 8(e)) and the 6-upsampling variant."""
    from seg2eye_b200.models import networks
    oopt = SimpleNamespace(**{**vars(ctx.oopt), **over})
    opt = SimpleNamespace(**{**vars(ctx.opt), **over})
    if "crop_size" in over:      # 'more' adds one upsampling: keep the 320x256 output (sw = 512 / 64 = 8, sh = 10)
        oopt.aspect_ratio = opt.aspect_ratio = 0.8
    sd = O.synth_state(O.generator_shapes(oopt), 77)
    seg = O.one_hot(ctx.batch["label"], 4)
    if "crop_size" in over:
        seg = torch.nn.functional.interpolate(seg, size=(640, 512), mode="nearest")
    w = O.synth_state({"w": (ctx.bs, 16)}, 5, scale=4.0)["w"]
    with torch.no_grad():
        ref = O.generator_forward({k: v.clone() for k, v in sd.items()}, seg, w, oopt)
    G = load(networks.SPADESTYLEGenerator(opt), sd).train()
    with torch.no_grad():
        out = G(seg.cuda(), w.cuda())
    assert out.shape == ref.shape
    assert rel(out, ref) < TOL_CHAIN, rel(out, ref)


def test_gan_loss_modes_vs_reference_fixture():
    """GANLoss (hinge | ls | original | w) on the device == the reference's GANLoss values recorded in
    tests/golden/ref_ganloss.npz (fp32 predictions: 1e-5), gradients == autograd through the oracle restatement."""
    from oracle.make_golden_ganloss import preds
    from seg2eye_b200.models import networks
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_ganloss.npz"))
    for key in ref.files:
        mode, real, for_d = key.rsplit("_", 2)
        real, for_d = bool(int(real)), bool(int(for_d))
        p_cpu = [[t.clone().requires_grad_() for t in d] for d in preds()]
        p_dev = [[t.cuda().requires_grad_() for t in d] for d in preds()]
        crit = networks.GANLoss(mode)
        got = crit(p_dev, real, for_discriminator=for_d)
        assert got.shape == (1,)
        np.testing.assert_allclose(got.detach().cpu().numpy(), ref[key], rtol=1e-5, atol=1e-6, err_msg=key)
        got.sum().backward()
        O.gan_loss(p_cpu, real, for_d, mode).sum().backward()
        for dc, dd in zip(p_cpu, p_dev):
            assert rel(dd[-1].grad, dc[-1].grad) < 1e-5, key
            assert dd[0].grad is None
    with pytest.raises(ValueError):
        networks.GANLoss("nope")


@pytest.mark.parametrize("mode", ["ls", "original"])
def test_training_iteration_other_gan_modes_vs_oracle(ctx, mode):
    """One full G + D iteration with gan_mode ls / original against the oracle trainer (losses within 2e-2)."""
    over = dict(gan_mode=mode)
    oopt = SimpleNamespace(**{**vars(ctx.oopt), **over})
    opt = SimpleNamespace(**{**vars(ctx.opt), **over})
    c2 = SimpleNamespace(oopt=oopt, opt=opt, bs=ctx.bs, seeds=ctx.seeds, batch=ctx.batch)
    tr = _make_trainer(c2)
    data = {k: v.clone() for k, v in ctx.batch.items()}
    tr.run_generator_one_step(data)
    tr.run_discriminator_one_step(data)
    ours = {k: float(v.reshape(-1)[0]) for k, v in tr.get_latest_losses().items()}
    sds = {n: O.synth_state(getattr(O, f + "_shapes")(oopt), ctx.seeds[n]) for n, f in (("G", "generator"), ("D", "discriminator"), ("E", "encoder"))}
    ot = O.OracleTrainer(sds["G"], sds["D"], sds["E"], oopt)
    ot.run_generator_one_step(ctx.batch)
    ot.run_discriminator_one_step(ctx.batch)
    ref = {k: float(v.reshape(-1)[0]) for k, v in {**ot.g_losses, **ot.d_losses}.items()}
    for k in ref:
        assert abs(ours[k] - ref[k]) <= TOL_LOSS * abs(ref[k]) + (2e-2 if k == "GAN" else 0.0), (k, ours[k], ref[k])


@pytest.mark.parametrize("fused", [True, False])
def test_training_iteration_with_and_without_fused_spade_conv_vs_oracle(ctx, fused):
    """One full G + D iteration with the training-mode fused gamma|beta-conv + modulation kernel (ops.SpadeConvFn, the
    default) and with the two-kernel path against the oracle trainer: losses within 2e-2, image within the chained bound."""
    from seg2eye_b200 import ops
    old = ops._state["fuse_spade_training"]
    ops._state["fuse_spade_training"] = fused
    try:
        tr = _make_trainer(ctx)
        data = {k: v.clone() for k, v in ctx.batch.items()}
        tr.run_generator_one_step(data)
        tr.run_discriminator_one_step(data)
    finally:
        ops._state["fuse_spade_training"] = old
    ours = {k: float(v.reshape(-1)[0]) for k, v in tr.get_latest_losses().items()}
    sds = {n: O.synth_state(getattr(O, f + "_shapes")(ctx.oopt), ctx.seeds[n]) for n, f in (("G", "generator"), ("D", "discriminator"), ("E", "encoder"))}
    ot = O.OracleTrainer(sds["G"], sds["D"], sds["E"], ctx.oopt)
    ot.run_generator_one_step(ctx.batch)
    ot.run_discriminator_one_step(ctx.batch)
    ref = {k: float(v.reshape(-1)[0]) for k, v in {**ot.g_losses, **ot.d_losses}.items()}
    for k in ref:
        assert abs(ours[k] - ref[k]) <= TOL_LOSS * abs(ref[k]) + (2e-2 if k == "GAN" else 0.0), (k, ours[k], ref[k])
    assert rel(tr.generated, ot.generated) < TOL_CHAIN


def test_eval_mode_inference_sweep_vs_oracle(ctx):
    """test.py runs the model in eval mode (BatchNorm running statistics, spectral-norm vectors frozen): the config-4
    sweep -- encode two style sets, interpolate, batch inference with `latent_style` -- against the oracle in eval mode;
    nothing in the state dicts may change."""
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(ctx.opt)
    sdG, sdE = O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"]), O.synth_state(O.encoder_shapes(ctx.oopt), ctx.seeds["E"])
    # eval mode uses the STORED u / v: random unit vectors would give sigma = u^T W v of arbitrary size and sign, i.e. a
    # network far outside its operating range; converge them first (what any trained checkpoint holds)
    for sd in (sdG, sdE):
        for k in [k for k in sd if k.endswith("weight_orig")]:
            wm = sd[k].reshape(sd[k].shape[0], -1)
            u, v = sd[k[:-5] + "_u"], sd[k[:-5] + "_v"]
            for _ in range(8):
                v.copy_(torch.nn.functional.normalize(wm.t() @ u, dim=0))
                u.copy_(torch.nn.functional.normalize(wm @ v, dim=0))
    load(m.netG, sdG)
    load(m.netE, sdE)
    m.eval()
    before = {k: v.clone() for k, v in m.netG.state_dict().items()}
    data = {k: v.clone() for k, v in ctx.batch.items()}
    w = m(data, mode="encode_only")
    with torch.no_grad():
        w_o = O.encode_w({k: v.clone() for k, v in sdE.items()}, ctx.batch["style_image"], ctx.oopt, training=False)
    assert rel(w, w_o) < TOL_ACT
    alphas = torch.linspace(0, 1, 5, device=w.device).view(-1, 1)
    wi = (1 - alphas) * w[0:1] + alphas * w[1:2]
    lab = ctx.batch["label"][0:1].repeat(5, 1, 1, 1)
    out = m({"label": lab, "style_image": ctx.batch["style_image"], "latent_style": wi.detach()}, mode="inference")
    with torch.no_grad():
        ref = O.generator_forward({k: v.clone() for k, v in sdG.items()}, O.one_hot(lab, 4), wi.detach().cpu(), ctx.oopt, training=False)
    assert out.shape == ref.shape and rel(out, ref) < TOL_CHAIN, rel(out, ref)
    after = m.netG.state_dict()
    assert all(torch.equal(before[k], after[k]) for k in before), "eval-mode inference changed buffers"


def test_optimizer_state_checkpoint_roundtrip(ctx, tmp_path):
    """SURVEY 8(f) row 4: trainer.save() also writes the Adam moments / step counts (`<epoch>_optim_{G,D}.pth`, keyed by
    parameter name); --continue_train restores networks AND optimizer state, so the resumed run continues the same
    trajectory instead of restarting Adam from zero moments (what the reference does)."""
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    opt = SimpleNamespace(**{**vars(ctx.opt), "checkpoints_dir": str(tmp_path), "name": "ck", "no_TTUR": True})
    c2 = SimpleNamespace(oopt=ctx.oopt, opt=opt, bs=ctx.bs, seeds=ctx.seeds, batch=ctx.batch)
    tr = _make_trainer(c2)
    data = {k: v.clone() for k, v in ctx.batch.items()}
    tr.run_generator_one_step(data)
    tr.run_discriminator_one_step(data)
    tr.save("latest")
    blob = torch.load(os.path.join(str(tmp_path), "ck", "latest_optim_G.pth"))
    assert blob["groups"][0]["step"] == 1.0 and "G.fc.weight" in blob["state"] and "E.fc_mu.weight" in blob["state"]
    assert "E.fc_var.weight" not in blob["state"]            # never receives a gradient, never gets Adam state
    opt2 = SimpleNamespace(**{**vars(opt), "continue_train": True})
    tr2 = Pix2PixTrainer(opt2)
    for (n1, p1), (n2, p2) in zip(tr.pix2pix_model.netG.named_parameters(), tr2.pix2pix_model.netG.named_parameters()):
        assert n1 == n2 and torch.equal(p1, p2)
        s1, s2 = tr.optimizer_G.state.get(p1), tr2.optimizer_G.state.get(p2)
        assert (not s1) == (not s2)
        if s1:
            assert torch.equal(s1["exp_avg"], s2["exp_avg"]) and torch.equal(s1["exp_avg_sq"], s2["exp_avg_sq"])
    assert float(tr2.optimizer_D.param_groups[0]["_s2e_state"][0]) == 1.0
    # both continue with the same second step (beta1 = 0.5 here, so the restored first moment matters)
    for t in (tr, tr2):
        d = {k: v.clone() for k, v in ctx.batch.items()}
        t.run_generator_one_step(d)
    a, b = tr.pix2pix_model.netG.state_dict(), tr2.pix2pix_model.netG.state_dict()
    assert rel(a["up_2.conv_0.weight_orig"], b["up_2.conv_0.weight_orig"]) < 1e-4
    assert rel(a["up_2.conv_0.weight_orig"] - ctx_sd(ctx)["up_2.conv_0.weight_orig"].cuda(),
               b["up_2.conv_0.weight_orig"] - ctx_sd(ctx)["up_2.conv_0.weight_orig"].cuda()) < 5e-2


def ctx_sd(ctx):
    return O.synth_state(O.generator_shapes(ctx.oopt), ctx.seeds["G"])


def test_training_trajectory_tracks_the_oracle(ctx):
    """Twelve full G + D iterations on a fixed batch (Adam with TTUR, all buffers advancing): the loss trajectory of the CUDA
    path must track the fp32 oracle's -- a drift in any kernel's gradient or in the optimiser would separate them within a
    few steps.  Bound: 5 % on the image-space L1 term (which falls steadily as the generator fits the target) and on the
    feature-matching term at every iteration, 5 % on the discriminator's hinge terms for the first eight."""
    tr = _make_trainer(ctx)
    sds = {n: O.synth_state(getattr(O, f + "_shapes")(ctx.oopt), ctx.seeds[n]) for n, f in (("G", "generator"), ("D", "discriminator"), ("E", "encoder"))}
    ot = O.OracleTrainer(sds["G"], sds["D"], sds["E"], ctx.oopt)
    ours, ref = [], []
    for it in range(12):
        data = {k: v.clone() for k, v in ctx.batch.items()}
        tr.run_generator_one_step(data)
        tr.run_discriminator_one_step(data)
        ot.run_generator_one_step(ctx.batch)
        ot.run_discriminator_one_step(ctx.batch)
        ours.append({k: float(v.reshape(-1)[0]) for k, v in tr.get_latest_losses().items()})
        ref.append({k: float(v.reshape(-1)[0]) for k, v in {**ot.g_losses, **ot.d_losses}.items()})
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out):
        import json
        json.dump({"ours": ours, "oracle": ref}, open(os.path.join(out, "trajectory_parity.json"), "w"), indent=1)
    # measured (gpurun_out/trajectory_parity.json): L1 within 1.2 %, feature matching within 2.5 % over all twelve iterations,
    # the hinge terms within 2 % for eight iterations; after that the two-player game itself becomes chaotic (the oracle run
    # on two different CPUs differs by 4 % in D/Fake at iteration 9), so the discriminator terms are only held that long
    for it, (a, b) in enumerate(zip(ours, ref)):
        for k in ("L1/weighted", "GAN_Feat"):
            assert abs(a[k] - b[k]) <= 5e-2 * abs(b[k]), (it, k, a[k], b[k])
        if it < 8:
            for k in ("D/Fake", "D/real"):
                assert abs(a[k] - b[k]) <= 5e-2 * abs(b[k]) + 2e-2, (it, k, a[k], b[k])
    assert ref[-1]["L1/weighted"] < 0.9 * ref[0]["L1/weighted"] and ours[-1]["L1/weighted"] < 0.9 * ours[0]["L1/weighted"]
