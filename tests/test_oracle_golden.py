"""Pin the CPU oracle (oracle/seg2eye_oracle.py) against outputs of the UNMODIFIED reference
recorded by oracle/make_golden.py (tests/golden/*.npz).  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import seg2eye_oracle as O
from oracle.make_golden import IMAGE_SUB

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(GOLD, "ref_small.npz")))


@pytest.fixture(scope="module")
def ints():
    return dict(np.load(os.path.join(GOLD, "ref_ints.npz")))


def cfg(gold):
    ngf, ndf, l1, bs = [int(x) for x in gold["meta_cfg"]]
    sG, sD, sE, sB = [int(x) for x in gold["meta_seeds"]]
    opt = O.make_opt(ngf=ngf, ndf=ndf, lambda_l1=float(l1))
    return opt, bs, dict(G=sG, D=sD, E=sE, batch=sB)


def sub(t, n=4096):
    f = t.detach().reshape(-1).double()
    step = max(1, f.numel() // n)
    return f[::step][:n].float().numpy(), np.array([float(f.norm()), float(f.mean()), f.numel()])


def close(a, b, tol=2e-4, atol=0.0):
    if torch.is_tensor(a):
        a = a.detach().double().numpy()
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    denom = max(np.linalg.norm(b.ravel()), 1e-12)
    err = np.linalg.norm((a - b).ravel())
    assert err <= tol * denom + atol * np.sqrt(a.size), (err / denom, err)


def test_integer_path_bit_exact(ints):
    seg = O.one_hot(torch.from_numpy(ints["label"]), 4)
    assert np.array_equal(seg.numpy().astype(np.uint8), ints["onehot"])
    for k, v in ints.items():
        if k.startswith("nearest_"):
            h, w = [int(s) for s in k.split("_")[1].split("x")]
            assert np.array_equal(O.nearest_resize(seg, (h, w)).numpy().astype(np.uint8), v), k
    seg2 = O.one_hot(torch.from_numpy(ints["rand_label"]), 4)
    assert np.array_equal(seg2.numpy().astype(np.uint8), ints["rand_onehot"])
    assert np.array_equal(O.nearest_resize(seg2, (9, 13)).numpy().astype(np.uint8), ints["rand_nearest_9x13"])


def test_encoder_generator_discriminator_forward(gold):
    opt, bs, seeds = cfg(gold)
    batch = O.synth_batch(opt, bs, seeds["batch"])
    seg = O.one_hot(batch["label"], 4)
    with torch.no_grad():
        sdE = O.synth_state(O.encoder_shapes(opt), seeds["E"])
        mu, logvar, feats = O.encoder_forward(sdE, batch["style_image"][0], opt)
        close(mu, gold["E_mu"])
        close(logvar, gold["E_logvar"])
        for i, f in enumerate(feats):
            s, st = sub(f)
            close(s, gold["E_feat%d_sub" % i])
            close(st, gold["E_feat%d_stat" % i])
        close(sdE["layer0.0.weight_u"], gold["E_layer0_u_after"], 1e-5)
        sdE = O.synth_state(O.encoder_shapes(opt), seeds["E"])
        w = O.encode_w(sdE, batch["style_image"], opt)
        close(w, gold["w"])

        sdG = O.synth_state(O.generator_shapes(opt), seeds["G"])
        taps = {}
        fake = O.generator_forward(sdG, seg, w, opt, taps=taps)
        s, st = sub(fake, IMAGE_SUB)
        close(s, gold["G_fake_sub"])
        close(st, gold["G_fake_stat"])
        for name in ("fc", "head_0", "head_0.norm_0", "G_middle_1", "up_0", "up_1", "up_3"):
            t = taps[name]
            if name.endswith("norm_0"):
                continue  # oracle tap is post-activation; the reference hook is pre-activation
            s, st = sub(t)
            close(s, gold["G_tap_%s_sub" % name])
            close(st, gold["G_tap_%s_stat" % name])
        for k in ("head_0.norm_0.spade.param_free_norm.running_mean", "up_3.norm_1.spade.param_free_norm.running_var",
                  "up_2.conv_0.weight_u", "up_2.conv_s.weight_v"):
            close(sdG[k], gold["G_buf_" + k], 1e-4)
        assert int(sdG["up_3.norm_1.spade.param_free_norm.num_batches_tracked"]) == int(
            gold["G_buf_up_3.norm_1.spade.param_free_norm.num_batches_tracked"])

        sdD = O.synth_state(O.discriminator_shapes(opt), seeds["D"])
        both = torch.cat([torch.cat([seg, fake], 1), torch.cat([seg, batch["target"]], 1)], 0)
        douts = O.discriminator_forward(sdD, both, opt)
        for i, d in enumerate(douts):
            for j, t in enumerate(d):
                s, st = sub(t)
                close(s, gold["D_%d_%d_sub" % (i, j)])
                close(st, gold["D_%d_%d_stat" % (i, j)])
        close(douts[0][4], gold["D_0_4"])
        close(douts[1][4], gold["D_1_4"])


def test_two_training_iterations(gold):
    opt, bs, seeds = cfg(gold)
    torch.manual_seed(0)
    batch = O.synth_batch(opt, bs, seeds["batch"])
    tr = O.OracleTrainer(O.synth_state(O.generator_shapes(opt), seeds["G"]),
                         O.synth_state(O.discriminator_shapes(opt), seeds["D"]),
                         O.synth_state(O.encoder_shapes(opt), seeds["E"]), opt)
    for it in range(2):
        tr.run_generator_one_step(batch)
        tr.run_discriminator_one_step(batch)
        for k, v in {**tr.g_losses, **tr.d_losses}.items():
            # iteration 1 follows an Adam(beta1=0) update ~ lr*sign(g): fp32 summation-order noise in
            # tiny gradients flips update signs, so near-zero losses (GAN) need an absolute floor
            close(v.detach().reshape(-1), gold["step%d_loss_%s" % (it, k)], 1e-3, atol=0.0 if it == 0 else 5e-4)
        s, st = sub(tr.generated, IMAGE_SUB)
        key = "G_fake" if it == 0 else "step%d_generated" % it     # iteration 0 generates G_fake again
        close(s, gold[key + "_sub"], 1e-3)
        close(st, gold[key + "_stat"], 1e-3)
    post = dict(G=tr.sdG, D=tr.sdD, E=tr.sdE)
    n = 0
    for k, v in gold.items():
        if not k.startswith("post_"):
            continue
        net, name = k[5], k[7:]
        if name.endswith("_stat"):
            continue
        if name.endswith("_sub"):
            s, st = sub(post[net][name[:-4]])
            close(s, v, 2e-3)
            close(st, gold[k[:-4] + "_stat"], 2e-3)
        else:
            close(post[net][name].detach().double(), v, 2e-3)
        n += 1
    assert n >= 15


def test_gan_loss_modes_match_reference_ganloss():
    """oracle.gan_loss in all four gan_modes == the reference's GANLoss (fixture from oracle/make_golden_ganloss.py)."""
    from oracle.make_golden_ganloss import preds
    ref = np.load(os.path.join(GOLD, "ref_ganloss.npz"))
    p = preds()
    assert len(ref.files) == 15
    for key in ref.files:
        mode, real, for_d = key.rsplit("_", 2)
        got = O.gan_loss(p, bool(int(real)), bool(int(for_d)), mode)
        assert got.shape == (1,)
        np.testing.assert_allclose(got.numpy(), ref[key], rtol=1e-6, atol=1e-7, err_msg=key)


def _variant_names():
    from oracle.make_golden_variants import VARIANTS
    return sorted(VARIANTS)


@pytest.mark.parametrize("name", _variant_names())
def test_option_variants_one_iteration(name):
    """One G + D iteration of the oracle == the UNMODIFIED reference trainer for the option variants of SURVEY 8(f) rank 1
    (spadeinstance, extra up-sampling, max aggregation, L2 loss, ls / original / wgan GAN modes, no feature matching,
    no TTUR): losses, generated image and post-step weights / buffers (fixture: oracle/make_golden_variants.py)."""
    from oracle.make_golden import SEEDS, SMALL
    from oracle.make_golden_variants import VARIANTS
    ref = np.load(os.path.join(GOLD, "ref_variants.npz"))
    oopt = O.make_opt(**{**SMALL, **VARIANTS[name][1]})
    sds = dict(G=O.synth_state(O.generator_shapes(oopt), SEEDS["G"]), D=O.synth_state(O.discriminator_shapes(oopt), SEEDS["D"]),
               E=O.synth_state(O.encoder_shapes(oopt), SEEDS["E"]))
    batch = O.synth_batch(oopt, 2, SEEDS["batch"])
    bias0 = sds["D"]["discriminator_1.model4.0.bias"].clone()
    tr = O.OracleTrainer(sds["G"], sds["D"], sds["E"], oopt)
    tr.run_generator_one_step(batch)
    tr.run_discriminator_one_step(batch)
    losses = {**tr.g_losses, **tr.d_losses}
    keys = [k.split("|")[2] for k in ref.files if k.startswith(name + "|loss|")]
    assert sorted(keys) == sorted(losses), (keys, sorted(losses))
    for k in keys:
        np.testing.assert_allclose(losses[k].detach().reshape(-1).numpy(), ref["%s|loss|%s" % (name, k)], rtol=2e-4, atol=2e-5, err_msg=k)
    s, st = sub(tr.generated)
    close(s, ref[name + "|generated_sub"], tol=5e-4)
    close(st[:2], ref[name + "|generated_stat"][:2], tol=5e-4)
    close(sds["G"]["conv_img.weight"], ref[name + "|post_G_conv_img.weight"], tol=5e-4)
    close(sds["G"]["up_1.conv_0.weight_u"], ref[name + "|post_G_up_1.conv_0.weight_u"], tol=5e-4)
    bias = sds["D"]["discriminator_1.model4.0.bias"]
    if oopt.gan_mode == "w":
        # the Wasserstein loss does not change when every logit shifts by the same constant: the gradient of the logit head's
        # bias is zero up to summation-order rounding, which Adam's first step (lr * g / (|g| + eps)) turns into any move in
        # [-lr, lr] (the reference's machine recorded 0.76 lr, another CPU computes g == 0 exactly): only the bound is defined
        assert float((bias - bias0).abs().max()) <= tr.opt_D.param_groups[0]["lr"] * (1 + 1e-5)
    else:
        close(bias, ref[name + "|post_D_model4_bias"], tol=5e-4, atol=1e-7)


def _variant2_names():
    from oracle.make_golden_variants import VARIANTS2
    return sorted(VARIANTS2)


@pytest.mark.parametrize("name", _variant2_names())
def test_style_gram_openeds_losses_one_iteration(name):
    """The optional loss branches of compute_generator_loss (pix2pix_model.py:209-231: openEDS, style_w, style_feat, Gram;
    max / mean aggregation of the encoder features): oracle == the UNMODIFIED reference trainer, one G + D iteration
    (fixture: oracle/make_golden_variants.py --second)."""
    from oracle.make_golden import SEEDS, SMALL
    from oracle.make_golden_variants import VARIANTS2
    ref = np.load(os.path.join(GOLD, "ref_variants2.npz"))
    oopt = O.make_opt(**{**SMALL, **VARIANTS2[name][1]})
    sds = dict(G=O.synth_state(O.generator_shapes(oopt), SEEDS["G"]), D=O.synth_state(O.discriminator_shapes(oopt), SEEDS["D"]),
               E=O.synth_state(O.encoder_shapes(oopt), SEEDS["E"]))
    batch = O.synth_batch(oopt, 2, SEEDS["batch"])
    tr = O.OracleTrainer(sds["G"], sds["D"], sds["E"], oopt)
    tr.run_generator_one_step(batch)
    tr.run_discriminator_one_step(batch)
    losses = {**tr.g_losses, **tr.d_losses}
    keys = [k.split("|")[2] for k in ref.files if k.startswith(name + "|loss|") and not k.endswith("/raw")]
    assert sorted(keys) == sorted(losses), (keys, sorted(losses))
    for k in keys:
        np.testing.assert_allclose(losses[k].detach().reshape(-1).numpy(), ref["%s|loss|%s" % (name, k)], rtol=3e-4, atol=2e-5, err_msg=k)
    s, st = sub(tr.generated)
    close(s, ref[name + "|generated_sub"], tol=5e-4)
    # the style losses reach the ENCODER through both the real and the fake features: its weights after the step pin that
    close(sds["G"]["conv_img.weight"], ref[name + "|post_G_conv_img.weight"], tol=5e-4)
    close(sds["G"]["up_1.conv_0.weight_u"], ref[name + "|post_G_up_1.conv_0.weight_u"], tol=5e-4)


def test_validation_tail_bit_exact_vs_reference_fixture():
    """oracle.to_255_resized / mse_for_images / to_255 == the reference's ImageProcessor.to_255resized_imagebatch (cv2
    INTER_LINEAR in float64, *255, .int()) and MSECalculator on the fixture inputs: every integer pixel (SHA-256 of the
    full result) and the per-image errors (fixture: oracle/make_golden_tail.py)."""
    from oracle.make_golden_tail import CASES, digest, tail_inputs
    ref = np.load(os.path.join(GOLD, "ref_tail.npz"))
    for name in CASES:
        fake, target = tail_inputs(name)
        got = O.to_255_resized(fake)
        assert got.dtype == torch.int32 and got.shape == (fake.shape[0], 1, 640, 400)
        assert np.array_equal(got.numpy().reshape(-1)[::997].astype(np.uint8), ref[name + "|sub"]), name
        assert np.array_equal(digest(got.numpy()), ref[name + "|sha256"]), name
        np.testing.assert_allclose(O.mse_for_images(got, target).numpy(), ref[name + "|errors"], rtol=1e-6)
    rng = np.random.Generator(np.random.PCG64(77))
    a = torch.from_numpy(rng.uniform(-1, 1, size=(3, 1, 64, 48)).astype(np.float32))
    b = torch.from_numpy(rng.uniform(-1, 1, size=(3, 1, 64, 48)).astype(np.float32))
    assert np.array_equal(digest(O.to_255(a).numpy()), ref["tensors|sha256"])
    np.testing.assert_allclose(O.mse_for_images(O.to_255(a), O.to_255(b)).numpy(), ref["tensors|errors"], rtol=1e-6)


def test_spade_layer_with_35_classes_vs_reference_fixture():
    """BASELINE config 5 per-layer pin: oracle.spade == the reference's SPADE module (normalization.py:63-105) with
    label_nc = 35, BatchNorm and InstanceNorm statistics, output / input gradient / mlp_shared weight gradient / running_var
    (fixture: oracle/make_golden_spade35.py)."""
    from oracle.make_golden_spade35 import CASES, inputs
    ref = np.load(os.path.join(GOLD, "ref_spade35.npz"))
    for name, (cfg, c, nc, _) in CASES.items():
        x, seg, sd = inputs(name)
        sd = {"L." + k: v.clone() for k, v in sd.items()}
        for k, v in sd.items():
            if v.dtype == torch.float32 and "running" not in k:
                v.requires_grad_(True)
        xr = x.clone().requires_grad_()
        y = O.spade(sd, "L", xr, seg, instance="instance" in cfg)
        y.square().mean().backward()
        s, st = sub(y)
        close(s, ref[name + "|out_sub"], tol=2e-5)
        close(st[:2], ref[name + "|out_stat"][:2], tol=2e-5)
        close(sub(xr.grad)[0], ref[name + "|dx_sub"], tol=2e-4)
        close(sub(sd["L.mlp_shared.0.weight"].grad)[0], ref[name + "|dw_shared_sub"], tol=2e-4)
        if "batch" in cfg:
            close(sd["L.param_free_norm.running_var"], ref[name + "|running_var"], tol=1e-5)


def test_data_layer_bit_exact_vs_reference_fixture():
    """oracle.preprocess_sample == the reference's get_transform pipeline ('fixed' mode: cv2 nearest for the mask, PIL bicubic +
    ToTensor + Normalize for the images, optional flip; data/base_dataset.py:50-80 as used by data/openeds_dataset.py:82-119):
    every label and every float bit (SHA-256 of the full results; fixture: oracle/make_golden_data.py)."""
    from oracle.make_golden_data import CASES, data_inputs, digest
    ref = np.load(os.path.join(GOLD, "ref_data.npz"))
    for name, (crop, ar, flip) in CASES.items():
        mask, images = data_inputs(name)
        w, h = crop, round(crop / ar)
        lab, ims = O.preprocess_sample(mask, images, w, h, flip)
        ims = torch.stack(ims)
        assert tuple(ims.shape) == tuple(ref[name + "|shape"]) and lab.shape == (h, w)
        assert np.array_equal(lab.numpy().reshape(-1)[::397].astype(np.uint8), ref[name + "|label_sub"]), name
        assert np.array_equal(digest(lab.numpy().astype(np.uint8)), ref[name + "|label_sha"]), name
        assert np.array_equal(ims.numpy().reshape(-1)[::997], ref[name + "|images_sub"]), name
        assert np.array_equal(digest(ims.numpy().astype(np.float32)), ref[name + "|images_sha"]), name
