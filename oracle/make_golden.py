"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (/root/reference) on CPU.

Runs only in the build container (the reference checkout does not travel to the GPU box).
The reference is imported, never copied; three import shims that touch no arithmetic are
applied (SURVEY.md 8(c)): a stub `h5py`, `cv2.cv2`, and float Adam betas.

    python oracle/make_golden.py            # writes tests/golden/ref_small.npz, ref_ints.npz

Weights come from oracle.seg2eye_oracle.synth_state (portable numpy PCG64), so tests can
rebuild the identical state dicts from (shapes, seed) without shipping the weights.
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("S2E_REFERENCE", "/root/reference")
sys.path.insert(0, REPO)

from oracle import seg2eye_oracle as O  # noqa: E402

SMALL = dict(ngf=16, ndf=16, lambda_l1=10.0)   # 320x256, label_nc 4, w_dim 16, input_ns 4
SEEDS = dict(G=101, D=202, E=303, batch=404)
IMAGE_SUB = 16384   # samples kept of a generated 2x1x320x256 image


def import_reference():
    sys.dont_write_bytecode = True
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    import cv2
    cv2.cv2 = cv2
    sys.modules["cv2.cv2"] = cv2
    _Adam = torch.optim.Adam

    class AdamF(_Adam):
        def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), **kw):
            super().__init__(params, lr=lr, betas=(float(betas[0]), float(betas[1])), **kw)

    torch.optim.Adam = AdamF
    sys.path.insert(0, REF)


def ref_opt(tmp, extra):
    from options.train_options import TrainOptions
    argv = ["train.py", "--dataroot", "/nonexistent", "--gpu_ids", "-1", "--name", "golden",
            "--checkpoints_dir", tmp] + extra
    old = sys.argv
    sys.argv = argv
    try:
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            opt = TrainOptions().parse()
    finally:
        sys.argv = old
    return opt


def sub(t, n=4096):
    """Deterministic subsample of a tensor (strided) + its L2 norm and mean."""
    f = t.detach().reshape(-1).double()
    step = max(1, f.numel() // n)
    return f[::step][:n].float().numpy(), np.array([float(f.norm()), float(f.mean()), f.numel()], dtype=np.float64)


def main():
    import_reference()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    out_dir = os.path.join(REPO, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    tmp = tempfile.mkdtemp()

    oopt = O.make_opt(**SMALL)
    extra = ["--ngf", str(SMALL["ngf"]), "--ndf", str(SMALL["ndf"]), "--lambda_l1", str(SMALL["lambda_l1"]),
             "--batchSize", "2"]
    opt = ref_opt(tmp, extra)

    import contextlib, io
    from trainers.pix2pix_trainer import Pix2PixTrainer
    with contextlib.redirect_stdout(io.StringIO()):
        trainer = Pix2PixTrainer(opt)
    model = trainer.pix2pix_model

    # ---- identical weights in the reference modules -------------------------------
    shapes = dict(G=O.generator_shapes(oopt), D=O.discriminator_shapes(oopt), E=O.encoder_shapes(oopt))
    nets = dict(G=model.netG, D=model.netD, E=model.netE)
    for k, net in nets.items():
        ref_sd = net.state_dict()
        assert list(ref_sd.keys()) == list(shapes[k].keys()), (k, set(ref_sd) ^ set(shapes[k]))
        for name, t in ref_sd.items():
            assert tuple(t.shape) == tuple(shapes[k][name]), (name, t.shape, shapes[k][name])
        net.load_state_dict(O.synth_state(shapes[k], SEEDS[k]))

    g = {}
    batch = O.synth_batch(oopt, 2, SEEDS["batch"])

    # ---- integer path -----------------------------------------------------------------
    ints = {}
    data = {k: v.clone() for k, v in batch.items()}
    seg, _, _ = model.preprocess_input(data)
    ints["label"] = batch["label"].numpy()
    ints["onehot"] = seg.numpy().astype(np.uint8)
    import torch.nn.functional as F
    for (h, w) in [(10, 8), (20, 16), (40, 32), (80, 64), (160, 128), (320, 256), (12, 7), (33, 50)]:
        r = F.interpolate(seg, size=(h, w), mode="nearest")
        ints["nearest_%dx%d" % (h, w)] = r.numpy().astype(np.uint8)
    # random-label worst case
    rng = np.random.Generator(np.random.PCG64(7))
    rl = torch.from_numpy(rng.integers(0, 4, size=(2, 1, 37, 53)).astype(np.uint8))
    d2 = {"label": rl.clone(), "style_image": batch["style_image"]}
    seg2, _, _ = model.preprocess_input(d2)
    ints["rand_label"] = rl.numpy()
    ints["rand_onehot"] = seg2.numpy().astype(np.uint8)
    ints["rand_nearest_9x13"] = F.interpolate(seg2, size=(9, 13), mode="nearest").numpy().astype(np.uint8)
    np.savez_compressed(os.path.join(out_dir, "ref_ints.npz"), **ints)

    # ---- module forwards (each on a fresh copy of the state so buffers start identical) --
    def fresh(k):
        nets[k].load_state_dict(O.synth_state(shapes[k], SEEDS[k]))

    model.train()
    with torch.no_grad():
        fresh("E")
        mu, logvar, feats = model.netE(batch["style_image"][0])
        g["E_mu"] = mu.numpy()
        g["E_logvar"] = logvar.numpy()
        for i, f in enumerate(feats):
            g["E_feat%d_sub" % i], g["E_feat%d_stat" % i] = sub(f)
        g["E_layer0_u_after"] = model.netE.state_dict()["layer0.0.weight_u"].numpy().copy()
        fresh("E")
        w = model.encode_w(batch["style_image"])[0]
        g["w"] = w.numpy()

        fresh("G")
        taps = {}
        hooks = []
        for name, mod in model.netG.named_modules():
            if name in ("fc", "head_0", "head_0.norm_0", "G_middle_1", "up_0", "up_1", "up_3", "up_3.norm_s", "up_3.norm_1"):
                hooks.append(mod.register_forward_hook(lambda m, i, o, name=name: taps.__setitem__(name, o.detach().clone())))
        fake = model.netG(seg, w)
        for h in hooks:
            h.remove()
        # images: a 1-in-10 subsample + norm / mean, which keeps the file small enough to commit
        g["G_fake_sub"], g["G_fake_stat"] = sub(fake, IMAGE_SUB)
        for name, t in taps.items():
            g["G_tap_%s_sub" % name], g["G_tap_%s_stat" % name] = sub(t)
        sdg = model.netG.state_dict()
        for k in ("head_0.norm_0.spade.param_free_norm.running_mean", "up_3.norm_1.spade.param_free_norm.running_var",
                  "up_3.norm_1.spade.param_free_norm.num_batches_tracked", "up_2.conv_0.weight_u", "up_2.conv_s.weight_v"):
            g["G_buf_" + k] = sdg[k].numpy().copy()

        fresh("D")
        both = torch.cat([torch.cat([seg, fake], 1), torch.cat([seg, batch["target"]], 1)], 0)
        douts = model.netD(both)
        for i, d in enumerate(douts):
            for j, t in enumerate(d):
                g["D_%d_%d_sub" % (i, j)], g["D_%d_%d_stat" % (i, j)] = sub(t)
        g["D_0_4"] = douts[0][4].numpy()
        g["D_1_4"] = douts[1][4].numpy()

    # ---- two full training iterations through the reference trainer ---------------------
    for k in nets:
        fresh(k)
    with contextlib.redirect_stdout(io.StringIO()):
        trainer = Pix2PixTrainer(opt)          # fresh optimizers
    for k, net in dict(G=trainer.pix2pix_model.netG, D=trainer.pix2pix_model.netD, E=trainer.pix2pix_model.netE).items():
        net.load_state_dict(O.synth_state(shapes[k], SEEDS[k]))
    for it in range(2):
        data = {k: v.clone() for k, v in batch.items()}
        trainer.run_generator_one_step(data)
        trainer.run_discriminator_one_step(data)
        for k, v in trainer.get_latest_losses().items():
            g["step%d_loss_%s" % (it, k)] = v.detach().reshape(-1).numpy().astype(np.float64)
        gen = trainer.get_latest_generated().detach()
        if it == 0:     # the first iteration generates from the same weights and inputs as the forward above: G_fake_*
            assert torch.equal(gen, fake)
        else:
            g["step%d_generated_sub" % it], g["step%d_generated_stat" % it] = sub(gen, IMAGE_SUB)
    m = trainer.pix2pix_model
    post = dict(G=m.netG.state_dict(), D=m.netD.state_dict(), E=m.netE.state_dict())
    for net, keys in dict(
        G=["fc.weight", "head_0.conv_0.weight_orig", "up_3.conv_s.weight_orig", "up_1.norm_0.spade.mlp_gamma.weight",
           "up_2.norm_1.adain.linear.weight", "conv_img.weight", "up_0.conv_1.weight_u",
           "up_3.norm_0.spade.param_free_norm.running_mean", "up_3.norm_0.spade.param_free_norm.num_batches_tracked"],
        D=["discriminator_0.model0.0.weight", "discriminator_1.model2.0.0.weight_orig", "discriminator_0.model3.0.0.weight_u",
           "discriminator_1.model4.0.bias"],
        E=["layer0.0.weight_orig", "layer5.0.weight_orig", "fc_mu.weight", "fc_var.weight", "layer3.0.weight_v"],
    ).items():
        for k in keys:
            t = post[net][k]
            if t.numel() <= 8192:
                g["post_%s_%s" % (net, k)] = t.numpy().copy()
            else:
                g["post_%s_%s_sub" % (net, k)], g["post_%s_%s_stat" % (net, k)] = sub(t)
    g["meta_seeds"] = np.array([SEEDS["G"], SEEDS["D"], SEEDS["E"], SEEDS["batch"]])
    g["meta_cfg"] = np.array([SMALL["ngf"], SMALL["ndf"], int(SMALL["lambda_l1"]), 2])
    np.savez_compressed(os.path.join(out_dir, "ref_small.npz"), **g)
    sz = {f: os.path.getsize(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}
    print("wrote", sz)
    for k in sorted(g):
        if "loss" in k:
            print(k, g[k])


if __name__ == "__main__":
    main()
