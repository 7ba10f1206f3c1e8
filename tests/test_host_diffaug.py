"""CPU-only checks of `--diff_augment` (differentiable augmentation of the D input): option parsing, rejection of unknown
ops and the canonical op order, which layout path `discriminate` takes, and the generator state in checkpoints
(`save`, `--continue_train` restore and fallback)."""
import argparse
import contextlib
import io
import os
from types import SimpleNamespace

import pytest
import torch

from oracle import seg2eye_oracle as O

NET_FILES = ("latest_net_G.pth", "latest_net_D.pth", "latest_net_E.pth")


def _opts(tmp, **kw):
    o = O.make_opt(ngf=8, ndf=8, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=str(tmp), name="da", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale")
    return SimpleNamespace(**d)


def _trainer(opt):
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    with contextlib.redirect_stdout(io.StringIO()):
        return Pix2PixTrainer(opt)


def _parser():
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    parser = argparse.ArgumentParser()
    parser.add_argument("--netG", default="spadestyle")
    parser.add_argument("--netD", default="multiscale")
    return Pix2PixModel.modify_commandline_options(parser, True)


def test_option_parses_in_canonical_order_and_rejects_unknown_ops(tmp_path):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    p = _parser()
    assert p.parse_args([]).diff_augment == ""
    assert p.parse_args(["--ema_decay", "0.5"]).ema_decay == 0.5      # registered next to --ema_decay
    for arg, want in (("color", "color"), ("cutout,translation", "translation,cutout"),
                      ("cutout, color ,translation", "color,translation,cutout"), ("translation", "translation")):
        assert p.parse_args(["--diff_augment", arg]).diff_augment == want
    for bad in ("colour", "color,flip", "translation,Cutout"):
        with contextlib.redirect_stderr(io.StringIO()), pytest.raises(SystemExit):
            p.parse_args(["--diff_augment", bad])
        with pytest.raises(ValueError):
            Pix2PixModel(_opts(tmp_path, diff_augment=bad))
    assert ops.parse_diff_augment("") == ((), 0)
    assert ops.parse_diff_augment("cutout,color") == (("color", "cutout"), 1 | 4)
    assert ops.parse_diff_augment("translation,color,cutout") == (("color", "translation", "cutout"), 7)


def test_state_exists_only_in_training_with_a_policy_and_leaves_the_layouts_alone(tmp_path):
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    torch.manual_seed(0)
    off = Pix2PixModel(_opts(tmp_path))
    after_off = torch.randint(0, 2 ** 30, (4,))
    torch.manual_seed(0)
    on = Pix2PixModel(_opts(tmp_path, diff_augment="color,cutout"))
    assert off.diffaug_state is None and off.diffaug_policy == 0
    st = on.diffaug_state
    assert st.dtype == torch.int64 and st.shape == (2,) and int(st[1]) == 0
    assert on.diffaug_ops == ("color", "cutout")
    # the default path consumes no random numbers of its own: today's initialisation stream is unchanged
    torch.manual_seed(0)
    Pix2PixModel(_opts(tmp_path))
    assert torch.equal(torch.randint(0, 2 ** 30, (4,)), after_off)
    for net in ("netG", "netD", "netE"):
        assert list(getattr(on, net).state_dict()) == list(getattr(off, net).state_dict())
    assert list(on.state_dict()) == list(off.state_dict())
    with contextlib.redirect_stdout(io.StringIO()):
        on.save("latest")
        test_time = Pix2PixModel(_opts(tmp_path, diff_augment="color", isTrain=False))
    assert test_time.diffaug_state is None


@pytest.mark.parametrize("policy", ["", "translation", "color,translation,cutout"])
def test_discriminate_augments_only_in_training_with_a_policy(tmp_path, policy, monkeypatch):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(_opts(tmp_path, diff_augment=policy))
    seen = []

    class Plain:
        @staticmethod
        def apply(seg, fake, real, cpad):
            seen.append(("plain", cpad))
            return torch.zeros(2 * seg.shape[0], seg.shape[2], seg.shape[3], cpad)

    class Aug:
        @staticmethod
        def apply(seg, fake, real, cpad, params, pol):
            seen.append(("aug", cpad, params, pol))
            return torch.zeros(2 * seg.shape[0], seg.shape[2], seg.shape[3], cpad)

    draws = []

    def draw(state, B, index_offset, H, W):
        draws.append((state, B, index_offset, H, W))
        return torch.full((B, 6), float(len(draws)))

    monkeypatch.setattr(ops, "MakeDInputFn", Plain)
    monkeypatch.setattr(ops, "MakeDInputAugFn", Aug)
    monkeypatch.setattr(ops, "diffaug_draw", draw)
    monkeypatch.setattr(m.netD, "forward_nhwc", lambda x: [[x[:, :1, :1, 0]]])
    seg, img = torch.zeros(3, 4, 8, 6), torch.zeros(3, 1, 8, 6)
    for training in (True, False):
        m.train(training)
        seen.clear()
        draws.clear()
        fake, real = m.discriminate(seg, img, img)
        assert fake[0][0].shape[0] == 3 and real[0][0].shape[0] == 3
        if policy and training:
            assert [s[0] for s in seen] == ["aug"] and seen[0][1] == 16
            assert seen[0][3] == m.diffaug_policy and seen[0][2] is not None
            assert len(draws) == 1 and draws[0][0] is m.diffaug_state and draws[0][1:] == (3, 0, 8, 6)
        else:
            assert seen == [("plain", 16)] and draws == []


def test_save_writes_the_generator_state_and_continue_train_restores_it(tmp_path):
    opt = _opts(tmp_path, diff_augment="translation,cutout")
    tr = _trainer(opt)
    st = tr.pix2pix_model.diffaug_state
    st.copy_(torch.tensor([-1234567890123456789, 2 ** 33 + 5]))
    tr.save("latest")
    d = os.path.join(opt.checkpoints_dir, opt.name)
    blob = torch.load(os.path.join(d, "latest_optim_D.pth"))
    assert blob["diffaug"] == {"seed": -1234567890123456789, "counter": 2 ** 33 + 5}
    assert "diffaug" not in torch.load(os.path.join(d, "latest_optim_G.pth"))
    # the network files are those of a run without the option, key for key and value for value
    nets_on = {f: torch.load(os.path.join(d, f)) for f in NET_FILES}
    opt_off = _opts(tmp_path)
    opt_off.name = "off"
    tr_off = _trainer(opt_off)
    m, m_off = tr.pix2pix_model, tr_off.pix2pix_model
    for net, net_off in ((m.netG, m_off.netG), (m.netD, m_off.netD), (m.netE, m_off.netE)):
        net_off.load_state_dict(net.state_dict())
    tr_off.save("latest")
    d_off = os.path.join(opt_off.checkpoints_dir, opt_off.name)
    assert sorted(os.listdir(d_off)) == sorted(os.listdir(d))
    assert "diffaug" not in torch.load(os.path.join(d_off, "latest_optim_D.pth"))
    for f, sd in nets_on.items():
        sd_off = torch.load(os.path.join(d_off, f))
        assert list(sd) == list(sd_off) and all(torch.equal(sd[k], sd_off[k]) for k in sd)
    # --continue_train restores seed and counter ...
    opt.continue_train = True
    st2 = _trainer(opt).pix2pix_model.diffaug_state
    assert st2.tolist() == [-1234567890123456789, 2 ** 33 + 5]
    # ... and a checkpoint without the entry (written with the option off) leaves a fresh seed at counter 0
    opt_off.continue_train, opt_off.diff_augment = True, "color"
    st3 = _trainer(opt_off).pix2pix_model.diffaug_state
    assert st3 is not None and int(st3[1]) == 0
