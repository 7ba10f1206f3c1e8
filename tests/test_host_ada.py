"""CPU-only checks of `--diff_augment_p` / `--ada_target` / `--ada_interval` / `--ada_kimg`: option parsing, range checks and
the dependency on `--diff_augment`, the default probability, which layout path `discriminate` takes, the `ada/*` entries of
the loss log, and the controller state in the `diffaug` checkpoint entry (`save`, `--continue_train` restore and fallback)."""
import argparse
import contextlib
import io
import os
from types import SimpleNamespace

import pytest
import torch

from oracle import seg2eye_oracle as O


def _opts(tmp, **kw):
    o = O.make_opt(ngf=8, ndf=8, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=str(tmp), name="ada", no_vgg_loss=True, lambda_openeds=0.0,
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


def test_options_parse_with_range_checks():
    p = _parser()
    a = p.parse_args([])
    assert (a.diff_augment_p, a.ada_target, a.ada_interval, a.ada_kimg) == (None, 0.0, 4, 500.0)
    a = p.parse_args(["--diff_augment", "color", "--diff_augment_p", "0.25", "--ada_target", "0.6", "--ada_interval", "8",
                      "--ada_kimg", "100"])
    assert (a.diff_augment_p, a.ada_target, a.ada_interval, a.ada_kimg) == (0.25, 0.6, 8, 100.0)
    for args in (["--diff_augment_p", "-0.1"], ["--diff_augment_p", "1.5"], ["--diff_augment_p", "nan"],
                 ["--ada_target", "1"], ["--ada_target", "-0.2"], ["--ada_target", "x"], ["--ada_interval", "0"],
                 ["--ada_interval", "2.5"], ["--ada_kimg", "0"], ["--ada_kimg", "inf"]):
        with contextlib.redirect_stderr(io.StringIO()), pytest.raises(SystemExit):
            p.parse_args(["--diff_augment", "color"] + args)


def test_probability_needs_a_policy_and_defaults_by_ada(tmp_path):
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    for kw in (dict(diff_augment_p=0.5), dict(ada_target=0.6), dict(diff_augment_p=1.0)):
        with pytest.raises(ValueError, match="--diff_augment"):
            Pix2PixModel(_opts(tmp_path, **kw))
    for kw in (dict(diff_augment_p=2.0), dict(ada_target=1.0), dict(ada_interval=0), dict(ada_kimg=-1.0)):
        with pytest.raises(ValueError):
            Pix2PixModel(_opts(tmp_path, diff_augment="color", **kw))
    plain = Pix2PixModel(_opts(tmp_path, diff_augment="color"))
    assert plain.diffaug_p == 1.0 and plain.ada_target == 0 and plain.ada_state is None
    explicit_one = Pix2PixModel(_opts(tmp_path, diff_augment="color", diff_augment_p=1.0))
    assert explicit_one.ada_state is None
    fixed = Pix2PixModel(_opts(tmp_path, diff_augment="color", diff_augment_p=0.4))
    assert fixed.ada_state is not None and float(fixed.ada_state["p"]) == 0.4
    ada = Pix2PixModel(_opts(tmp_path, diff_augment="color,cutout", ada_target=0.6))
    st = ada.ada_state
    assert float(st["p"]) == 0.0 and ada.ada_interval == 4 and ada.ada_kimg == 500.0
    assert st["p"].dtype == st["acc"].dtype == st["record"].dtype == torch.float64
    assert st["acc"].shape == (6,) and st["record"].shape == (5,) and st["pos"].dtype == torch.int32    # num_D = 2
    assert float(Pix2PixModel(_opts(tmp_path, diff_augment="color", ada_target=0.6, diff_augment_p=0.3)).ada_state["p"]) == 0.3
    assert list(ada.state_dict()) == list(plain.state_dict())


@pytest.mark.parametrize("kw,path", [(dict(), "aug"), (dict(diff_augment_p=1.0), "aug"), (dict(diff_augment_p=0.5), "masked"),
                                     (dict(ada_target=0.6), "masked")])
def test_discriminate_takes_the_masked_path_only_below_one_or_with_ada(tmp_path, monkeypatch, kw, path):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(_opts(tmp_path, diff_augment="translation", **kw))
    seen = []

    class Aug:
        @staticmethod
        def apply(seg, fake, real, cpad, params, pol):
            seen.append("aug")
            return torch.zeros(2 * seg.shape[0], seg.shape[2], seg.shape[3], cpad)

    class Masked:
        @staticmethod
        def apply(seg, fake, real, cpad, params, opmask, pol):
            seen.append(("masked", opmask))
            return torch.zeros(2 * seg.shape[0], seg.shape[2], seg.shape[3], cpad)

    draws = []
    monkeypatch.setattr(ops, "MakeDInputAugFn", Aug)
    monkeypatch.setattr(ops, "MakeDInputAugMaskedFn", Masked)
    monkeypatch.setattr(ops, "diffaug_draw", lambda st, B, o, H, W: torch.zeros(B, 6))
    monkeypatch.setattr(ops, "diffaug_draw_p", lambda st, p, B, o, H, W: (draws.append(p), (torch.zeros(B, 6), torch.zeros(B)))[1])
    monkeypatch.setattr(m.netD, "forward_nhwc", lambda x: [[x[:, :1, :1, 0]]])
    seg, img = torch.zeros(2, 4, 8, 6), torch.zeros(2, 1, 8, 6)
    m.train()
    m.discriminate(seg, img, img)
    if path == "aug":
        assert seen == ["aug"] and draws == []
    else:
        assert seen[0][0] == "masked" and draws == [m.ada_state["p"]]


def test_ada_entries_go_to_the_loss_log_not_the_loss_dict(tmp_path, monkeypatch):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(_opts(tmp_path, diff_augment="color", ada_target=0.6))
    y = torch.tensor([[0.5, -1.0], [2.0, 0.0], [3.0, -0.5], [1.0, 4.0]]).view(4, 1, 1, 2)    # [fake ; real] logits, B = 2
    logits = [[y], [y * -2]]      # num_D = 2

    def discriminate(seg, fake, real):
        m._last_d_out = logits
        return m.divide_pred(logits)
    monkeypatch.setattr(ops, "sign_sum", lambda x: torch.sign(x.float()).sum().reshape(1))   # S2E_RED_SIGN's result
    monkeypatch.setattr(m, "discriminate", discriminate)
    monkeypatch.setattr(m, "generate_fake", lambda seg, style: (torch.zeros(2, 1, 8, 6),))
    monkeypatch.setattr(type(m.criterionGAN), "__call__", lambda self, pred, real, for_discriminator=True: torch.zeros(()))
    losses = m.compute_discriminator_loss(torch.zeros(2, 4, 8, 6), None, torch.zeros(2, 1, 8, 6))
    assert set(losses) == {"D/Fake", "D/real"}
    assert m.ada_state["record"].tolist() == [2.0, 4.0, -2.0, 4.0, 2.0]   # real half [3, -0.5, 1, 4] and its negation
    log = m.get_loss_log()
    assert set(log) == {"ada/p", "ada/rt"} and float(log["ada/p"]) == 0.0 and float(log["ada/rt"]) == 0.0
    m.ada_state["p"].fill_(0.125)
    assert float(m.get_loss_log()["ada/p"]) == 0.125     # the live value


def test_checkpoint_round_trip_and_fallback(tmp_path):
    opt = _opts(tmp_path, diff_augment="translation,cutout", ada_target=0.6)
    tr = _trainer(opt)
    st = tr.pix2pix_model.ada_state
    st["p"].fill_(0.3125)
    st["acc"].copy_(torch.tensor([3.0, 40.0, -5.0, 10.0, 8.0, 0.4375], dtype=torch.float64))
    st["pos"].fill_(3)
    tr.save("latest")
    d = os.path.join(opt.checkpoints_dir, opt.name)
    blob = torch.load(os.path.join(d, "latest_optim_D.pth"))["diffaug"]
    assert blob["p"] == 0.3125 and blob["acc"] == [3.0, 40.0, -5.0, 10.0, 8.0, 0.4375] and blob["pos"] == 3
    assert set(blob) == {"seed", "counter", "p", "acc", "pos"}
    opt.continue_train = True
    st2 = _trainer(opt).pix2pix_model.ada_state
    assert float(st2["p"]) == 0.3125 and st2["acc"].tolist() == [3.0, 40.0, -5.0, 10.0, 8.0, 0.4375] and int(st2["pos"]) == 3
    # a fixed probability is an option, not state: the entry is today's, and restoring keeps the option's value
    opt_p = _opts(tmp_path, diff_augment="color", diff_augment_p=0.5)
    opt_p.name = "fixed"
    tr_p = _trainer(opt_p)
    tr_p.save("latest")
    assert set(torch.load(os.path.join(opt_p.checkpoints_dir, "fixed", "latest_optim_D.pth"))["diffaug"]) == {"seed", "counter"}
    # a checkpoint written before (or without ADA) restores the seed and counter and leaves the start state
    opt_old = _opts(tmp_path, diff_augment="color")
    opt_old.name = "old"
    tr_old = _trainer(opt_old)
    tr_old.pix2pix_model.diffaug_state[1] = 17
    tr_old.save("latest")
    opt_old.continue_train, opt_old.ada_target = True, 0.6
    m = _trainer(opt_old).pix2pix_model
    assert int(m.diffaug_state[1]) == 17
    assert float(m.ada_state["p"]) == 0.0 and not m.ada_state["acc"].any() and int(m.ada_state["pos"]) == 0
