"""CPU-only checks of `--diff_augment xflip,geometric`: parsing and the canonical op order, `flip` still rejected, which
layout path `discriminate` takes (and that p is held on the device for the new ops), the unchanged checkpoint entry, and
the H, W >= 2 check of the geometric warp."""
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
             which_epoch="latest", checkpoints_dir=str(tmp), name="geom", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netG="spadestyle", netD="multiscale")
    return SimpleNamespace(**d)


def _parser():
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    parser = argparse.ArgumentParser()
    parser.add_argument("--netG", default="spadestyle")
    parser.add_argument("--netD", default="multiscale")
    return Pix2PixModel.modify_commandline_options(parser, True)


def test_new_ops_parse_in_canonical_order_and_flip_is_still_rejected(tmp_path):
    from seg2eye_b200 import _lib as L
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    assert [n for n, _ in ops.DIFFAUG_OPS] == ["color", "xflip", "geometric", "translation", "cutout"]
    assert (L.DIFFAUG_XFLIP, L.DIFFAUG_GEOMETRIC, L.DIFFAUG_GEOM_RECORD) == (8, 16, 8)
    p = _parser()
    for arg, want in (("geometric", "geometric"), ("xflip", "xflip"), ("cutout,geometric,xflip,color,translation",
                                                                      "color,xflip,geometric,translation,cutout"),
                      ("translation, geometric", "geometric,translation")):
        assert p.parse_args(["--diff_augment", arg]).diff_augment == want
    assert ops.parse_diff_augment("geometric,xflip") == (("xflip", "geometric"), 8 | 16)
    assert ops.parse_diff_augment("cutout,xflip,color,geometric,translation") == (
        ("color", "xflip", "geometric", "translation", "cutout"), 31)
    for bad in ("flip", "color,flip", "yflip", "geometry", "rotate90", "xint", "Geometric"):
        with contextlib.redirect_stderr(io.StringIO()), pytest.raises(SystemExit):
            p.parse_args(["--diff_augment", bad])
        with pytest.raises(ValueError):
            Pix2PixModel(_opts(tmp_path, diff_augment=bad))


def test_new_ops_hold_p_on_the_device_and_leave_the_state_dicts_alone(tmp_path):
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    plain = Pix2PixModel(_opts(tmp_path, diff_augment="color,translation"))
    assert plain.ada_state is None
    for policy in ("xflip", "geometric", "color,xflip,geometric,translation,cutout"):
        m = Pix2PixModel(_opts(tmp_path, diff_augment=policy))
        assert m.ada_target == 0 and float(m.ada_state["p"]) == 1.0 and m.ada_state["p"].dtype == torch.float64
        assert list(m.state_dict()) == list(plain.state_dict())
    assert float(Pix2PixModel(_opts(tmp_path, diff_augment="geometric", diff_augment_p=0.25)).ada_state["p"]) == 0.25
    assert float(Pix2PixModel(_opts(tmp_path, diff_augment="geometric", ada_target=0.6)).ada_state["p"]) == 0.0


@pytest.mark.parametrize("policy,kw,path", [("color,translation,cutout", {}, "aug"),
                                            ("color,translation,cutout", dict(diff_augment_p=0.5), "masked"),
                                            ("xflip", {}, "geom"), ("geometric,cutout", {}, "geom"),
                                            ("color,xflip,geometric", dict(ada_target=0.6), "geom")])
def test_discriminate_takes_the_geometric_path_exactly_with_a_new_op(tmp_path, monkeypatch, policy, kw, path):
    from seg2eye_b200 import ops
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    m = Pix2PixModel(_opts(tmp_path, diff_augment=policy, **kw))
    seen, draws = [], []

    def layout(name):
        class Fn:
            @staticmethod
            def apply(seg, *args):
                seen.append((name, args[-1]))
                return torch.zeros(2 * seg.shape[0], seg.shape[2], seg.shape[3], args[2])
        return Fn

    def draw_geom(st, p, B, o, H, W):
        draws.append(("geom", p, B, o, H, W))
        return torch.zeros(B, 6), torch.zeros(B, 8), torch.zeros(B, dtype=torch.int32)

    monkeypatch.setattr(ops, "MakeDInputAugFn", layout("aug"))
    monkeypatch.setattr(ops, "MakeDInputAugMaskedFn", layout("masked"))
    monkeypatch.setattr(ops, "MakeDInputAugGeomFn", layout("geom"))
    monkeypatch.setattr(ops, "diffaug_draw", lambda st, B, o, H, W: (draws.append(("plain",)), torch.zeros(B, 6))[1])
    monkeypatch.setattr(ops, "diffaug_draw_p", lambda st, p, B, o, H, W: (draws.append(("p", p)),
                                                                          (torch.zeros(B, 6), torch.zeros(B)))[1])
    monkeypatch.setattr(ops, "diffaug_draw_geom", draw_geom)
    monkeypatch.setattr(m.netD, "forward_nhwc", lambda x: [[x[:, :1, :1, 0]]])
    seg, img = torch.zeros(2, 4, 8, 6), torch.zeros(2, 1, 8, 6)
    m.train()
    m.discriminate(seg, img, img)
    assert seen == [(path, m.diffaug_policy)]
    want_draw = {"aug": "plain", "masked": "p", "geom": "geom"}[path]
    assert len(draws) == 1 and draws[0][0] == want_draw
    if path == "geom":
        assert draws[0][1] is m.ada_state["p"] and draws[0][2:] == (2, 0, 8, 6)
    m.eval()       # inference never augments
    seen.clear()
    monkeypatch.setattr(ops, "MakeDInputFn", layout("plain"))
    m.discriminate(seg, img, img)
    assert [s[0] for s in seen] == ["plain"]


def test_checkpoint_entry_is_unchanged_by_the_new_ops(tmp_path):
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    opt = _opts(tmp_path, diff_augment="xflip,geometric,cutout")
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    tr.pix2pix_model.diffaug_state.copy_(torch.tensor([987654321, 41]))
    tr.pix2pix_model.ada_state["p"].fill_(0.75)       # not state without ADA: neither saved nor restored
    tr.save("latest")
    blob = torch.load(os.path.join(opt.checkpoints_dir, opt.name, "latest_optim_D.pth"))["diffaug"]
    assert blob == {"seed": 987654321, "counter": 41}
    opt.continue_train = True
    with contextlib.redirect_stdout(io.StringIO()):
        m = Pix2PixTrainer(opt).pix2pix_model
    assert m.diffaug_state.tolist() == [987654321, 41] and float(m.ada_state["p"]) == 1.0


@pytest.mark.parametrize("hw", [(1, 8), (8, 1), (1, 1)])
def test_geometric_needs_two_by_two_maps(hw):
    from seg2eye_b200 import _lib as L
    from seg2eye_b200 import ops
    H, W = hw
    B, nc = 2, 4
    seg, img = torch.zeros(B, nc, H, W), torch.zeros(B, 1, H, W)
    params, geom = torch.zeros(B, 6), torch.zeros(B, 8)
    mask = torch.full((B,), 31, dtype=torch.int32)
    for policy in (L.DIFFAUG_GEOMETRIC, L.DIFFAUG_GEOMETRIC | L.DIFFAUG_XFLIP | L.DIFFAUG_COLOR):
        with pytest.raises(ValueError, match="2 x 2"):
            ops.MakeDInputAugGeomFn.apply(seg, img, img, 16, params, mask, geom, policy)
