"""CPU-only checks of `--ema_decay` (exponential moving average of the G and E weights): option parsing and range, the
EMA nets' construction and state_dict layout, the checkpoint files they add, --continue_train restore and fallback, and
test-time loading of the averaged generator."""
import argparse
import os
from types import SimpleNamespace

import pytest
import torch

from oracle import seg2eye_oracle as O

BASE_FILES = {"latest_net_G.pth", "latest_net_D.pth", "latest_net_E.pth", "latest_optim_G.pth", "latest_optim_D.pth"}


def _opts(tmp, **kw):
    netG = kw.pop("netG", "spadestyle")
    o = O.make_opt(ngf=8, ndf=8, netG=netG, **kw)
    d = vars(o).copy()
    d.update(gpu_ids=[], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir=str(tmp), name="ema", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netD="multiscale")
    return o, SimpleNamespace(**d)


def _trainer(opt):
    import contextlib
    import io
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    with contextlib.redirect_stdout(io.StringIO()):
        return Pix2PixTrainer(opt)


def _same(a, b):
    sa, sb = a.state_dict(), b.state_dict()
    return list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)


def test_ema_decay_option_parses_and_rejects_values_outside_unit_interval(tmp_path):
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    parser = argparse.ArgumentParser()
    parser.add_argument("--netG", default="spadestyle")
    parser.add_argument("--netD", default="multiscale")
    Pix2PixModel.modify_commandline_options(parser, True)
    assert parser.parse_args([]).ema_decay == 0.0
    assert parser.parse_args(["--ema_decay", "0.999"]).ema_decay == 0.999
    for bad in (1.0, -0.1, 1.5, float("nan")):
        _, opt = _opts(tmp_path, ema_decay=bad)
        with pytest.raises(ValueError):
            Pix2PixModel(opt)


def test_ema_off_creates_no_nets_and_saves_todays_files(tmp_path):
    _, opt = _opts(tmp_path, ema_decay=0.0)
    tr = _trainer(opt)
    m = tr.pix2pix_model
    assert m.netG_ema is None and m.netE_ema is None
    assert tr.optimizer_G.ema is None and tr.optimizer_G.ema_buffers == []
    assert not any("ema" in k for k in m.state_dict())
    tr.save("latest")
    assert set(os.listdir(os.path.join(opt.checkpoints_dir, opt.name))) == BASE_FILES


@pytest.mark.parametrize("netG", ["spadestyle", "spade"])
def test_ema_nets_are_frozen_copies_with_the_live_layout(tmp_path, netG):
    oopt, opt = _opts(tmp_path, ema_decay=0.9, netG=netG)
    _, opt_off = _opts(tmp_path, ema_decay=0.0, netG=netG)
    tr = _trainer(opt)
    m = tr.pix2pix_model
    assert type(m.netG_ema) is type(m.netG) and _same(m.netG_ema, m.netG)
    if netG == "spade":
        assert m.netE is None and m.netE_ema is None
    else:
        assert type(m.netE_ema) is type(m.netE) and _same(m.netE_ema, m.netE)
    nets = [n for n in (m.netG_ema, m.netE_ema) if n is not None]
    assert all(not p.requires_grad for n in nets for p in n.parameters())
    # G / E carry exactly the reference layout, with EMA on and off
    m_off = _trainer(opt_off).pix2pix_model
    oopt.netG = netG
    for mm in (m, m_off):
        assert list(mm.netG.state_dict()) == list(O.generator_shapes(oopt))
        if mm.netE is not None:
            assert list(mm.netE.state_dict()) == list(O.encoder_shapes(oopt))
    # the G optimizer covers every G+E parameter with its average, and every buffer pair
    opt_G = tr.optimizer_G
    live = [p for n in (m.netG, m.netE) if n is not None for p in n.parameters()]
    assert opt_G.ema_decay == 0.9 and set(map(id, opt_G.ema)) == set(map(id, live))
    assert all(opt_G.ema[p].shape == p.shape and opt_G.ema[p] is not p for p in live)
    n_bufs = sum(len(list(n.buffers())) for n in nets)
    assert len(opt_G.ema_buffers) == n_bufs and tr.optimizer_D.ema is None


def test_ema_checkpoints_continue_train_and_test_time(tmp_path):
    from seg2eye_b200.models import networks
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    _, opt = _opts(tmp_path, ema_decay=0.99)
    tr = _trainer(opt)
    m = tr.pix2pix_model
    with torch.no_grad():   # averages that differ from G / E
        for n in (m.netG_ema, m.netE_ema):
            for t in list(n.parameters()) + list(n.buffers()):
                t.add_(1)
    tr.save("latest")
    d = os.path.join(opt.checkpoints_dir, opt.name)
    assert set(os.listdir(d)) == BASE_FILES | {"latest_net_G_ema.pth", "latest_net_E_ema.pth"}
    # the files carry G's / E's keys and load strictly into fresh networks
    for tag, define, ema in (("G", networks.define_G, m.netG_ema), ("E", networks.define_E, m.netE_ema)):
        sd = torch.load(os.path.join(d, "latest_net_%s_ema.pth" % tag))
        fresh = define(opt)
        fresh.load_state_dict(sd, strict=True)
        assert _same(fresh, ema)
    # --continue_train restores the averages bitwise ...
    opt.continue_train = True
    m2 = _trainer(opt).pix2pix_model
    assert _same(m2.netG_ema, m.netG_ema) and _same(m2.netE_ema, m.netE_ema)
    assert _same(m2.netG, m.netG) and not _same(m2.netG_ema, m2.netG)
    # ... and starts them from the loaded G / E when a run without EMA wrote the checkpoint
    for tag in ("G", "E"):
        os.remove(os.path.join(d, "latest_net_%s_ema.pth" % tag))
    m3 = _trainer(opt).pix2pix_model
    assert _same(m3.netG_ema, m.netG) and _same(m3.netE_ema, m.netE)
    # test time with --ema_decay > 0 (restored by --load_from_opt_file): G comes from the _ema file
    tr.save("7")
    opt_t = SimpleNamespace(**{**vars(opt), "isTrain": False, "continue_train": False, "which_epoch": "7"})
    mt = Pix2PixModel(opt_t)
    assert _same(mt.netG, m.netG_ema) and mt.netG_ema is None and mt.netD is None
    opt_t.ema_decay = 0.0
    assert _same(Pix2PixModel(opt_t).netG, m.netG)


def test_load_state_dict_into_live_nets_restarts_the_averages(tmp_path):
    _, opt = _opts(tmp_path, ema_decay=0.9)
    tr = _trainer(opt)
    m = tr.pix2pix_model
    g_ptrs = [p.data_ptr() for p in m.netG_ema.parameters()]
    sd = {k: v.clone() + (0.5 if v.is_floating_point() else 3) for k, v in m.netG.state_dict().items()}
    m.netG.load_state_dict(sd)
    assert not _same(m.netG_ema, m.netG)
    m.sync_ema()         # what the next G step, inference or save does first
    assert _same(m.netG_ema, m.netG) and _same(m.netE_ema, m.netE)
    assert [p.data_ptr() for p in m.netG_ema.parameters()] == g_ptrs     # in place: captured graphs stay valid
    with torch.no_grad():
        next(m.netG_ema.parameters()).add_(1)
    tr.reset_optimizers()
    assert _same(m.netG_ema, m.netG)
