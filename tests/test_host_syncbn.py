"""CPU-only checks of `--norm_G spectralspadesyncbatch3x3` (SyncBatchNorm inside SPADE): it parses for both generators,
its networks carry exactly the state_dict of `spectralspadebatch3x3`, and checkpoints load across the two with
strict=True."""
from types import SimpleNamespace

import pytest
import torch

from oracle import seg2eye_oracle as O


def _opts(**kw):
    o = O.make_opt(**kw)
    d = vars(o).copy()
    d.update(gpu_ids=[], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir="/tmp/s2e_ckpt", name="t", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netD="multiscale")
    d.setdefault("netG", "spadestyle")
    return o, SimpleNamespace(**d)


def _spades(net):
    from seg2eye_b200.models.networks.normalization import SPADE
    return [m for m in net.modules() if isinstance(m, SPADE)]


@pytest.mark.parametrize("netG", ["spadestyle", "spade"])
def test_syncbatch_state_dict_equals_batch(netG):
    from seg2eye_b200.models import networks
    extra = dict(netG=netG) if netG == "spade" else {}
    oopt, opt_b = _opts(ngf=8, ndf=8, norm_G="spectralspadebatch3x3", **extra)
    _, opt_s = _opts(ngf=8, ndf=8, norm_G="spectralspadesyncbatch3x3", **extra)
    opt_b.netG = opt_s.netG = netG
    torch.manual_seed(0)
    g_b = networks.define_G(opt_b)
    torch.manual_seed(1)
    g_s = networks.define_G(opt_s)
    sp_b, sp_s = _spades(g_b), _spades(g_s)
    assert sp_s and len(sp_s) == len(sp_b)
    assert all(s.sync for s in sp_s) and not any(s.sync for s in sp_b)
    sd_b, sd_s = g_b.state_dict(), g_s.state_dict()
    assert list(sd_b) == list(sd_s)
    for k in sd_b:
        assert sd_b[k].shape == sd_s[k].shape and sd_b[k].dtype == sd_s[k].dtype, k
    # the layout is the reference's (whose SPADE with `spectralspadebatch3x3` reads the same checkpoint)
    oopt.netG = netG
    shapes = O.generator_shapes(oopt)
    assert set(sd_s) == set(shapes)
    for k, shp in shapes.items():
        assert tuple(sd_s[k].shape) == tuple(shp), k
    # checkpoints cross over in both directions, strictly
    g_s.load_state_dict(sd_b, strict=True)
    for k, v in g_s.state_dict().items():
        assert torch.equal(v, sd_b[k]), k
    g_b.load_state_dict({k: v.clone() + (1 if v.is_floating_point() else 0) for k, v in sd_s.items()}, strict=True)
    for k, v in g_b.state_dict().items():
        assert torch.equal(v, sd_s[k] + (1 if v.is_floating_point() else 0)), k


@pytest.mark.parametrize("cfg,ks", [("spadesyncbatch3x3", 3), ("spadesyncbatch5x5", 5), ("spadebatch3x3", 3)])
def test_spade_parses_syncbatch(cfg, ks):
    from seg2eye_b200.models.networks.normalization import SPADE
    from seg2eye_b200.models.networks.layers import BatchNorm2dStats
    s = SPADE(cfg, 16, 4)
    assert isinstance(s.param_free_norm, BatchNorm2dStats) and not s.per_sample
    assert s.sync == ("sync" in cfg)
    assert s.mlp_gamma.cfg.kh == ks and s.mlp_shared[0].cfg.kh == ks


def test_sync_applies_only_to_training_batch_statistics_across_ranks():
    from seg2eye_b200 import _lib as L, ops
    cfg = ops.NormCfg(False, L.ACT_NONE, True, 0.1, 1e-5, True)
    # one process (no process group): the plain batch-statistics path, same kernels and launches as `spadebatch`
    assert not ops.synced(cfg)
    assert ops.NormCfg(False, L.ACT_NONE, True, 0.1, 1e-5).sync is False
