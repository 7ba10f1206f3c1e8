"""Autograd operators over the seg2eye_b200 C ABI.

Internal convention: activations are contiguous bf16 tensors shaped (B, H, W, C) ("NHWC").  The module
layer (models/networks) exposes the reference's logical-NCHW interface through zero-copy permuted views.
Every arithmetic step calls one of our CUDA kernels through ctypes; torch is used for memory, streams and
the autograd graph only.
"""
import contextlib
import os
from collections import namedtuple

import torch

from . import _lib as L
from . import parallel

BF16 = torch.bfloat16
F32 = torch.float32

HEAD_ON_TC = os.environ.get("S2E_HEAD_TC", "0") == "1"   # A/B knob: PatchGAN head zero-padded onto the tcgen05 kernels
ConvCfg = namedtuple("ConvCfg", "kh kw stride pad act relu_in cin_pad cout_pad in_act", defaults=(False, 0, 0, 0))
# cin_pad: the activations carry cin_pad >= Cin channels (zero padded), packed weights get zero columns for them
# relu_in: the input of this convolution is the output of a ReLU whose backward is fused into our data-gradient epilogue
# in_act:  activation applied to the input as the kernel loads it (LeakyReLU in front of conv_img, generator.py:97-98);
#          its backward rides in the data-gradient kernel (mask = the saved pre-activation input).  Thin-layer kernels only
# cout_pad: run a layer with very few output channels (the 1-channel PatchGAN head, K = 8192) on the tensor-core kernels
#           with its output channels zero-padded to cout_pad; the caller sees the first Cout channels only

_state = {"force_impl": None, "weights_epoch": 0, "skip_wgrad": False,
          # SpadeConvFn: training-mode gamma|beta conv + modulation in one kernel (measured on B200, round 1: 111.3 ->
          # 109.3 ms/step; it lost 2 ms before the fused epilogue became its own template instantiation, when its
          # extra registers spilled in EVERY forward kernel).  S2E_FUSE_SPADE_TRAINING=0 restores the two-kernel path.
          "fuse_spade_training": __import__("os").environ.get("S2E_FUSE_SPADE_TRAINING", "1") == "1"}


def set_halo(on, base_offset=False):
    """3x3 / stride-1 tensor-core convolutions with an N tile <= 128 take the halo-tile kernel (library debug key 6)."""
    _state["halo"] = bool(on)
    L.call("s2e_debug_set", 6, (1 if on else 0) | (2 if base_offset else 0))


def halo_on():
    if "halo" not in _state:      # first use: S2E_DEBUG may have set the key at load time; S2E_HALO=0/1 overrides
        import os
        env = os.environ.get("S2E_HALO")
        if env is not None:
            set_halo(env == "1")
        else:
            _state["halo"] = any(item.strip() in ("6=1", "6=3") for item in os.environ.get("S2E_DEBUG", "").split(","))
    return _state["halo"]


def bump_weights_epoch():
    """Called whenever parameters are modified behind torch's back (our Adam kernel)."""
    _state["weights_epoch"] += 1


@contextlib.contextmanager
def force_impl(impl):
    """Testing aid: route every tap-convolution through one implementation (L.IMPL_TC / L.IMPL_SIMT)."""
    old = _state["force_impl"]
    _state["force_impl"] = impl
    try:
        yield
    finally:
        _state["force_impl"] = old


@contextlib.contextmanager
def skip_weight_grads():
    """Skip weight-gradient kernels of convolutions run inside (their parameters receive no .grad).
    Used for the discriminator inside the generator step, whose parameter gradients the reference computes
    and then discards (pix2pix_trainer.py:39 zeroes them before the next use)."""
    old = _state["skip_wgrad"]
    _state["skip_wgrad"] = True
    try:
        yield
    finally:
        _state["skip_wgrad"] = old


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# ---- optional per-kernel timing with CUDA events on the launching stream (bench.py roofline numbers)
_prof = None


def profile_begin():
    global _prof
    _prof = {"tc": [], "norm": [], "normb": []}


def profile_end(dump_path=None):
    global _prof
    p, _prof = _prof, None
    torch.cuda.synchronize()
    agg = {}
    for kind in p:
        for a, b, w, tag in p[kind]:
            e = agg.setdefault((kind, tag), [0, 0.0, 0.0])
            e[0] += 1
            e[1] += a.elapsed_time(b)
            e[2] += w
    if dump_path:
        with open(dump_path, "w") as f:
            f.write("kind\ttag\tlaunches\tms_total\twork\trate(TFLOP/s|GB/s)\n")
            for (kind, tag), (n, ms, w) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                rate = (w / 1e12 if kind == "tc" else w / 1e9) / (ms / 1e3) if ms > 0 else 0
                f.write("%s\t%s\t%d\t%.3f\t%.4g\t%.1f\n" % (kind, tag, n, ms, w, rate))
    out = {"by_tag": agg}
    for kind, key in (("tc", "flop"), ("norm", "bytes"), ("normb", "bytes")):
        rows = [v for (k, _), v in agg.items() if k == kind]
        out[kind + "_ms"] = sum(v[1] for v in rows)
        out[kind + "_" + key] = float(sum(v[2] for v in rows))
        out[kind + "_n"] = sum(v[0] for v in rows)
    return out


def _timed_call(kind, work, name, *args, tag=""):
    if _prof is None:
        return L.call(name, *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    L.call(name, *args)
    e1.record()
    _prof[kind].append((e0, e1, work, tag))


def _pick(tc_ok):
    if _state["force_impl"] is not None:
        if _state["force_impl"] == L.IMPL_TC and not tc_ok:
            return L.IMPL_SIMT
        return _state["force_impl"]
    return L.IMPL_TC if tc_ok else L.IMPL_SIMT


# ------------------------------------------------------------------------------------------------ conv
_taps_cache = {}


def conv_taps(cfg):
    key = (cfg.kh, cfg.kw, cfg.stride, cfg.pad)
    if key not in _taps_cache:
        _taps_cache[key] = L.packed_taps(*key)
    return _taps_cache[key]


def conv_out_hw(cfg, hi, wi):
    return (hi + 2 * cfg.pad - cfg.kh) // cfg.stride + 1, (wi + 2 * cfg.pad - cfg.kw) // cfg.stride + 1


_FTILE = tuple(int(v) for v in os.environ["S2E_FTILE"].split(",")) if os.environ.get("S2E_FTILE") else None
_KTILE = tuple(int(v) for v in os.environ["S2E_KTILE"].split(",")) if os.environ.get("S2E_KTILE") else None


def _desc(B, Hi, Wi, Cin, Ho, Wo, Cout, taps, act, negate=False):
    d = L.ConvDesc()
    d.B, d.Hi, d.Wi, d.Cin, d.Ho, d.Wo, d.Cout = B, Hi, Wi, Cin, Ho, Wo, Cout
    d.ntaps = len(taps)
    for i, (dy, dx) in enumerate(taps):
        d.tap_dy[i] = -dy if negate else dy
        d.tap_dx[i] = -dx if negate else dx
    d.act = act
    if _KTILE:      # bring-up aid: S2E_KTILE="w,h,b" overrides the weight-gradient kernels' pixel tile
        d.ktile_w, d.ktile_h, d.ktile_b = _KTILE
    if _FTILE:      # bring-up aid: S2E_FTILE="w,h,b" overrides the forward / data-gradient kernels' pixel tile
        d.tile_w, d.tile_h, d.tile_b = _FTILE
    return d


# ---- packed bf16 weight copies ---------------------------------------------------------------------------------
# One registry for every packed copy (tap-major forward / transposed layouts, im2col'd mlp_shared weights).  A copy is
# stale when one of its master weights changed: torch's own version counter (copy_, load_state_dict, init) or the
# per-tensor counter our Adam kernel bumps (it writes through raw pointers).  Stale copies are re-packed in ONE
# multi-tensor launch: right after an optimizer step (optim.Adam.step -> repack_stale()), or lazily at first use.
import ctypes as _C
import weakref as _weakref


class _PackEntry:
    __slots__ = ("refs", "cfg", "transposed", "im2col", "buf", "ver")

    def weights(self):
        ws = [r() for r in self.refs]
        return None if any(w is None for w in ws) else ws


_pack_cache = {}


def _master_version(weights):
    return (tuple(w._version for w in weights), tuple(w.data_ptr() for w in weights),
            tuple(getattr(w, "_s2e_ver", 0) for w in weights), _state["weights_epoch"])


def mark_updated(params):
    """Our Adam kernel changed these tensors behind torch's back."""
    for p_ in params:
        p_._s2e_ver = getattr(p_, "_s2e_ver", 0) + 1


def pack_on_use(tensors):
    """Leave the packed copies of these tensors out of repack_stale(): they are re-packed only when a forward reads them
    after their versions changed (mark_updated(), copy_, load_state_dict).  For the EMA nets (--ema_decay), whose
    weights every G step changes but only an inference with them reads: re-packing them in the training step would
    double its re-pack traffic."""
    for t in tensors:
        t._s2e_pack_on_use = True


def _pack_jobs(entry, weights):
    jobs = []
    if entry.im2col:       # weights = (weight,) or (weight, bias): the bias goes to column 63
        w = weights[0].detach()
        j = L.PackJob()
        j.w_oihw, j.out_bf16, j.Cout, j.Cin, j.im2col3x3 = w.data_ptr(), entry.buf.data_ptr(), w.shape[0], w.shape[1], 1
        j.bias = weights[1].detach().data_ptr() if len(weights) > 1 else None
        return [j]
    cfg = entry.cfg
    ctot = max(sum(w.shape[0] for w in weights), cfg.cout_pad)
    off = 0
    for w in weights:
        wd = w.detach()
        assert wd.is_contiguous() and wd.dtype == F32
        j = L.PackJob()
        j.w_oihw, j.out_bf16 = wd.data_ptr(), entry.buf.data_ptr()
        j.Cout, j.Cin, j.kh, j.kw, j.stride, j.pad = wd.shape[0], wd.shape[1], cfg.kh, cfg.kw, cfg.stride, cfg.pad
        j.transposed, j.Cout_total, j.co_offset, j.cin_pad, j.im2col3x3 = int(entry.transposed), ctot, off, cfg.cin_pad, 0
        jobs.append(j)
        off += wd.shape[0]
    return jobs


def _run_pack_jobs(jobs):
    if jobs:
        arr = (L.PackJob * len(jobs))(*jobs)
        L.call("s2e_pack_weight_multi", arr, len(jobs), L.stream())


def repack_pending():
    """True when weights were changed wholesale since the last re-pack (bump_weights_epoch: checkpoint load,
    load_state_dict, state restore).  Cheap enough to ask before every CUDA-graph replay, whose captured kernels read the
    packed copies without any host-side staleness check."""
    return _state.get("packed_epoch") != _state["weights_epoch"]


def repack_stale():
    """Re-pack every registered copy whose master weights changed (except those of pack_on_use tensors), in one launch
    per 40 tensors."""
    _state["packed_epoch"] = _state["weights_epoch"]
    jobs, dead = [], []
    for key, e in _pack_cache.items():
        ws = e.weights()
        if ws is None:
            dead.append(key)
            continue
        if any(getattr(w, "_s2e_pack_on_use", False) for w in ws):
            continue
        ver = _master_version(ws)
        if ver != e.ver:
            jobs += _pack_jobs(e, ws)
            e.ver = ver
    for key in dead:
        del _pack_cache[key]
    _run_pack_jobs(jobs)
    return len(jobs)


def _packed(key, weights, cfg, transposed, im2col, numel):
    e = _pack_cache.get(key)
    if e is not None and not all(r() is w for r, w in zip(e.refs, weights)):
        e = None     # a recycled id(): never alias a dead tensor's copy
    ver = _master_version(weights)
    if e is not None and e.ver == ver:
        return e.buf
    if e is None:
        e = _PackEntry()
        e.refs = tuple(_weakref.ref(w) for w in weights)
        e.cfg, e.transposed, e.im2col = cfg, transposed, im2col
        # zero-filled ONCE: padding slots (stride-2 phases, cin_pad / im2col filler columns) are never written again
        e.buf = torch.zeros(numel, dtype=BF16, device=weights[0].device)
        _pack_cache[key] = e
    _run_pack_jobs(_pack_jobs(e, weights))
    e.ver = ver
    return e.buf


def packed_weights(weights, cfg, transposed):
    """bf16 tap-major copy of one or more OIHW fp32 master weights (concatenated along Cout)."""
    key = (tuple(id(w) for w in weights), transposed, cfg.kh, cfg.kw, cfg.stride, cfg.pad, cfg.cin_pad, cfg.cout_pad)
    cin_eff = max(weights[0].shape[1], cfg.cin_pad)
    cinp = cin_eff * 4 if cfg.stride == 2 else cin_eff
    ctot = max(sum(w.shape[0] for w in weights), cfg.cout_pad)
    return _packed(key, weights, cfg, transposed, False, len(conv_taps(cfg)) * ctot * cinp)


def packed_weight_im2col(weight, bias=None):
    """bf16 [Cout][64] copy of a thin 3x3 weight (k = (r*3+s)*C + c) for the im2col'd segmap GEMM; `bias` fills
    columns 62 | 63 (lo | hi part), which multiply the two constant-one channels of the im2col'd segmap."""
    ws = (weight,) if bias is None else (weight, bias)
    return _packed((tuple(id(w) for w in ws), "im2col"), ws, None, False, True, weight.shape[0] * 64)


def space_to_depth(x):
    B, H, W, Cc = x.shape
    y = torch.empty(B, (H + 1) // 2, (W + 1) // 2, 4 * Cc, dtype=BF16, device=x.device)
    L.call("s2e_space_to_depth", L.ptr(x), B, H, W, Cc, L.ptr(y), L.stream())
    return y


def channel_sums(x2d_c, B, HW, Cc):
    """fp32 per-channel sum over all pixels of an NHWC bf16 tensor (bias gradients).  s2e_norm_stats accumulates shifted
    data, sum (x - p) with the pivot p = first pixel: the plain sum is that + n * p."""
    acc = torch.empty(3 * Cc, dtype=torch.float64, device=x2d_c.device)
    L.call("s2e_norm_stats", L.ptr(x2d_c), B, HW, Cc, 0, L.ptr(acc), L.stream())
    return (acc[:Cc] + float(B * HW) * acc[2 * Cc:]).to(F32)


class TapConvFn(torch.autograd.Function):
    """y = act(inv_sigma * conv(x, W) + b) [+ res] for one or several weights concatenated along Cout.

    res (optional, shaped like y): residual added in the tcgen05 epilogue (architecture.py:44 `x_s + dx`).
    cfg.cout_pad: a layer with fewer than 8 output channels and a long reduction (the PatchGAN logit head) runs on the
    tensor-core kernels with zero-padded output channels; forward returns the first Cout channels of the padded result."""

    @staticmethod
    def forward(ctx, x, cfg, sn, n_w, res, *wb):
        weights, biases = wb[:n_w], wb[n_w:]
        x = _c(x)
        assert x.dtype == BF16 and x.dim() == 4
        B, Hi, Wi, Cin = x.shape
        assert Cin == max(weights[0].shape[1], cfg.cin_pad), "channel mismatch: x has %d, weight expects %d" % (
            Cin, max(weights[0].shape[1], cfg.cin_pad))
        xs = space_to_depth(x) if cfg.stride == 2 else x
        _, His, Wis, Cinp = xs.shape
        Ho, Wo = conv_out_hw(cfg, Hi, Wi)
        Cout = sum(w.shape[0] for w in weights)
        padded = cfg.cout_pad > Cout and Cinp % 64 == 0 and cfg.cout_pad % 8 == 0 and _pick(True) == L.IMPL_TC
        if not padded:
            cfg = cfg._replace(cout_pad=0)
        Cp = cfg.cout_pad if padded else Cout
        taps = conv_taps(cfg)
        wp = packed_weights(weights, cfg, False)
        bias = None
        if len(biases):
            bias = biases[0].detach() if len(biases) == 1 else torch.cat([b.detach() for b in biases])
        inv_sigma = sn[2] if sn is not None else None
        y = torch.empty(B, Ho, Wo, Cp, dtype=BF16, device=x.device)
        d = _desc(B, His, Wis, Cinp, Ho, Wo, Cp, taps, cfg.act)
        d.bias_n = Cout
        d.in_act = cfg.in_act
        impl = _pick(Cinp % 64 == 0 and Cp % 8 == 0)
        assert cfg.in_act == L.ACT_NONE or (impl == L.IMPL_SIMT and cfg.stride == 1), "in_act: thin CUDA-core layers only"
        fuse_res = res is not None and impl == L.IMPL_TC and Cp % 64 == 0
        if res is not None:
            res = _c(res)
            assert cfg.act == L.ACT_NONE and not padded and res.shape == y.shape and res.dtype == BF16
            if fuse_res:
                d.residual = L.ptr(res)
        flops = 2.0 * B * Ho * Wo * Cout * weights[0].shape[1] * cfg.kh * cfg.kw
        if impl == L.IMPL_TC:
            _timed_call("tc", flops, "s2e_tapconv_fwd", d, L.ptr(xs), L.ptr(wp), L.ptr(bias), L.ptr(inv_sigma), L.ptr(y), impl, L.stream(),
                        tag="fwd B%d %dx%d Cin%d Cout%d T%d" % (B, Ho, Wo, Cinp, Cp, len(taps)))
        else:
            L.call("s2e_tapconv_fwd", d, L.ptr(xs), L.ptr(wp), L.ptr(bias), L.ptr(inv_sigma), L.ptr(y), impl, L.stream())
        if res is not None and not fuse_res:
            L.call("s2e_add", L.ptr(y), L.ptr(res), y.numel(), L.ptr(y), L.stream())
        ctx.flops = flops
        ctx.cfg, ctx.sn, ctx.n_w, ctx.n_b = cfg, sn, n_w, len(biases)
        ctx.in_shape = (B, Hi, Wi, Cin)
        ctx.weights = weights
        ctx.cout, ctx.cp = Cout, Cp
        ctx.skip_wgrad = _state["skip_wgrad"]
        ctx.save_for_backward(xs, y if cfg.act != L.ACT_NONE else None)
        return y[..., :Cout] if padded else y

    @staticmethod
    def backward(ctx, dy):
        cfg, sn, weights = ctx.cfg, ctx.sn, ctx.weights
        xs, y = ctx.saved_tensors
        dy = _c(dy)
        B, Hi, Wi, Cin = ctx.in_shape
        _, His, Wis, Cinp = xs.shape
        _, Ho, Wo, _ = dy.shape
        Cout_true, Cout = ctx.cout, ctx.cp
        taps = conv_taps(cfg)
        st = L.stream()
        dy_true = dy
        if Cout != Cout_true:     # zero-padded output channels: the kernels see the padded gradient
            dy = torch.zeros(B, Ho, Wo, Cout, dtype=BF16, device=dy.device)
            dy[..., :Cout_true].copy_(dy_true)
        if cfg.act != L.ACT_NONE:
            dpre = torch.empty_like(dy)
            L.call("s2e_act_bwd", L.ptr(dy), L.ptr(y), dy.numel(), cfg.act, L.ptr(dpre), st)
        else:
            dpre = dy
        inv_sigma = sn[2] if sn is not None else None
        dx = None
        if ctx.needs_input_grad[0]:
            wpt = packed_weights(weights, cfg, True)
            dd = _desc(B, Ho, Wo, Cout, His, Wis, Cinp, taps, L.ACT_NONE, negate=True)
            if cfg.relu_in:
                assert cfg.stride == 1 and Cinp % 64 == 0
                dd.relu_mask = L.ptr(xs)   # x = relu(.) > 0 exactly where the ReLU passed gradient
            if cfg.in_act != L.ACT_NONE:   # gradient w.r.t. the PRE-activation input: act'(x) * conv^T(dy)
                dd.relu_mask = L.ptr(xs)
                dd.mask_slope = 0.2 if cfg.in_act == L.ACT_LRELU else 0.0
            dxs = torch.empty(B, His, Wis, Cinp, dtype=BF16, device=dy.device)
            impl = _pick(Cout % 64 == 0 and Cinp % 8 == 0)
            if impl == L.IMPL_TC:
                _timed_call("tc", ctx.flops, "s2e_tapconv_fwd", dd, L.ptr(dpre), L.ptr(wpt), None, L.ptr(inv_sigma), L.ptr(dxs), impl, st,
                            tag="dgrad B%d %dx%d Cin%d Cout%d T%d" % (B, His, Wis, Cout, Cinp, len(taps)))
            else:
                L.call("s2e_tapconv_fwd", dd, L.ptr(dpre), L.ptr(wpt), None, L.ptr(inv_sigma), L.ptr(dxs), impl, st)
            if cfg.stride == 2:
                dx = torch.empty(B, Hi, Wi, Cin, dtype=BF16, device=dy.device)
                L.call("s2e_depth_to_space", L.ptr(dxs), B, Hi, Wi, Cin, L.ptr(dx), st)
            else:
                dx = dxs
        need_w = [ctx.needs_input_grad[5 + i] and not ctx.skip_wgrad for i in range(ctx.n_w)]
        need_b = [ctx.needs_input_grad[5 + ctx.n_w + i] and not ctx.skip_wgrad for i in range(ctx.n_b)]
        gw = [None] * ctx.n_w
        gb = [None] * ctx.n_b
        if any(need_w):
            dwp = torch.zeros(len(taps) * Cout * Cinp, dtype=F32, device=dy.device)
            d = _desc(B, His, Wis, Cinp, Ho, Wo, Cout, taps, L.ACT_NONE)
            d.in_act = cfg.in_act
            impl = _pick(Cinp >= 64 and Cout >= 64 and Cinp % 8 == 0 and Cout % 8 == 0)
            if impl == L.IMPL_TC:
                _timed_call("tc", ctx.flops, "s2e_tapconv_wgrad", d, L.ptr(xs), L.ptr(dpre), L.ptr(dwp), impl, st,
                            tag="wgrad B%d %dx%d Cin%d Cout%d T%d" % (B, Ho, Wo, Cinp, Cout, len(taps)))
            else:
                L.call("s2e_tapconv_wgrad", d, L.ptr(xs), L.ptr(dpre), L.ptr(dwp), impl, st)
            dot = torch.empty(1, dtype=F32, device=dy.device) if sn is not None else None
            off = 0
            for i, w in enumerate(weights):
                if need_w[i]:
                    g = torch.empty_like(w)
                    L.call("s2e_unpack_wgrad", L.ptr(dwp), w.shape[0], w.shape[1], cfg.kh, cfg.kw, cfg.stride, cfg.pad,
                           Cout, off, cfg.cin_pad, L.ptr(w.detach()), L.ptr(sn[0]) if sn else None, L.ptr(sn[1]) if sn else None,
                           L.ptr(inv_sigma), L.ptr(dot), L.ptr(g), 0, st)
                    gw[i] = g
                off += w.shape[0]
        if any(need_b):
            # per-channel sums left on the gradient tensor by its producer (SPADE+Style backward) -- valid only if the tensor
            # was not accumulated into since (autograd may add a second gradient in place: the version counter moves)
            pre = getattr(dy, '_s2e_chsum', None) if cfg.act == L.ACT_NONE else None
            if pre is not None and getattr(dy, '_s2e_chsum_ver', None) != (dy._version, dy.data_ptr()):
                pre = None
            if pre is not None and pre.numel() == Cout:
                _state["chsum_hits"] = _state.get("chsum_hits", 0) + 1
                sums = pre      # the producer of dy (SPADE+Style backward) already reduced it over the pixels
            elif Cout != Cout_true:
                sums = dy_true.float().sum(dim=(0, 1, 2))
            else:
                sums = channel_sums(dpre, B, Ho * Wo, Cout) if Cout % 8 == 0 else dpre.float().sum(dim=(0, 1, 2))
            off = 0
            for i in range(ctx.n_b):
                n = weights[i].shape[0]
                if need_b[i]:
                    gb[i] = sums[off:off + n].clone()
                off += n
        gres = dy_true if ctx.needs_input_grad[4] else None
        return (dx, None, None, None, gres) + tuple(gw) + tuple(gb)


def tap_conv(x, cfg, weights, biases=(), sn=None, residual=None):
    return TapConvFn.apply(x, cfg, sn, len(weights), residual, *weights, *biases)


_head_wd_cache = {}


def _head_dgrad_weight(weight):
    """[Cin][64] bf16 copy of a (1, Cin, kh, kw) head weight, column t = tap t (taps >= kh*kw zero): the weight of the 1x1
    convolution G (64 tap channels) -> dx.  The buffer is zero-filled once; each call refreshes the live columns."""
    ent = _head_wd_cache.get(id(weight))
    Cin, nt = weight.shape[1], weight.shape[2] * weight.shape[3]
    if ent is None or ent[0]() is not weight or ent[1].device != weight.device:
        buf = torch.zeros(Cin, 64, dtype=BF16, device=weight.device)
        _head_wd_cache[id(weight)] = ent = (_weakref.ref(weight), buf)
    ent[1][:, :nt].copy_(weight.detach()[0].reshape(Cin, nt))
    return ent[1]


def head_conv_ok(x, cfg, weight, sn=None):
    """Shapes HeadConvFn takes: one output channel, wide input, stride 1, at most 16 taps, no activation / spectral norm."""
    return (weight.shape[0] == 1 and cfg.stride == 1 and cfg.kh * cfg.kw <= 16 and weight.shape[1] % 64 == 0
            and 128 <= weight.shape[1] <= 1024 and x.shape[-1] == weight.shape[1] and cfg.act == L.ACT_NONE
            and cfg.in_act == L.ACT_NONE and sn is None and _state["force_impl"] is None)


class HeadConvFn(torch.autograd.Function):
    """PatchGAN logit head conv(x, W) + b with W of shape (1, Cin, kh, kw), stride 1 (discriminator.py:38) in tap-channel
    form: D[q][t] = x[q] . W[t] (the input is read once, CUDA cores, fp32), y[p] = sum_t D[p + tap_t][t] + b.  Backward:
    G[q][t] = dy[q - tap_t] (64 channels, kh*kw live), dx = G . W and dW = G^T . x as 1x1 convolutions on the tcgen05 kernels."""

    @staticmethod
    def forward(ctx, x, cfg, weight, bias):
        x = _c(x)
        B, Hi, Wi, Cin = x.shape
        Ho, Wo = conv_out_hw(cfg, Hi, Wi)
        taps = conv_taps(cfg)
        wp = packed_weights((weight,), cfg, False)          # [tap][1][Cin] bf16
        D = torch.empty(B * Hi * Wi, 16, dtype=F32, device=x.device)
        y = torch.empty(B, Ho, Wo, 1, dtype=BF16, device=x.device)
        # [fake ; real] batches: the sums behind GANLoss's hinge / Wasserstein terms ride in the gather kernel's epilogue
        signs = _state.get("sign_sums")
        signs = signs if B % 2 == 0 else None
        sums = torch.zeros(7 if signs is not None else 6, dtype=F32, device=x.device) if B % 2 == 0 else None
        d = _desc(B, Hi, Wi, Cin, Ho, Wo, 1, taps, L.ACT_NONE)
        st = L.stream()
        L.call("s2e_head_dots", L.ptr(x), L.ptr(wp), B * Hi * Wi, Cin, len(taps), L.ptr(D), st)
        b_ptr = L.ptr(bias.detach() if bias is not None else None)
        if signs is None:
            L.call("s2e_head_gather", d, L.ptr(D), b_ptr, None, L.ptr(y), L.ptr(sums), st)
        else:     # slot 6: sum sign(y) over the real half (head_sign_sums)
            L.call("s2e_head_gather_signs", d, L.ptr(D), b_ptr, None, L.ptr(y), L.ptr(sums), L.ptr(sums[6:]), st)
            signs[y.data_ptr()] = sums[6:]
        ctx.cfg, ctx.has_b = cfg, bias is not None
        ctx.skip_wgrad = _state["skip_wgrad"]
        ctx.save_for_backward(x, weight)
        if sums is None:
            return y, None
        ctx.mark_non_differentiable(sums)
        return y, sums

    @staticmethod
    def backward(ctx, dy, _dsums=None):
        x, weight = ctx.saved_tensors
        cfg = ctx.cfg
        dy = _c(dy)
        B, Hi, Wi, Cin = x.shape
        _, Ho, Wo, _ = dy.shape
        taps = conv_taps(cfg)
        st = L.stream()
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[2] and not ctx.skip_wgrad
        need_b = ctx.has_b and ctx.needs_input_grad[3] and not ctx.skip_wgrad
        dx = gw = gb = None
        if need_x or need_w:
            G = torch.empty(B, Hi, Wi, 64, dtype=BF16, device=dy.device)
            L.call("s2e_head_scatter", _desc(B, Hi, Wi, Cin, Ho, Wo, 1, taps, L.ACT_NONE), L.ptr(dy), L.ptr(G), st)
            one = [(0, 0)]
            flops = 2.0 * B * Ho * Wo * Cin * len(taps)
        if need_x:
            wd = _head_dgrad_weight(weight)
            dx = torch.empty(B, Hi, Wi, Cin, dtype=BF16, device=dy.device)
            _timed_call("tc", flops, "s2e_tapconv_fwd", _desc(B, Hi, Wi, 64, Hi, Wi, Cin, one, L.ACT_NONE), L.ptr(G), L.ptr(wd), None, None,
                        L.ptr(dx), L.IMPL_TC, st, tag="dgrad-head B%d %dx%d Cin64 Cout%d T1" % (B, Hi, Wi, Cin))
        if need_w:
            dwp = torch.zeros(64, Cin, dtype=F32, device=dy.device)
            _timed_call("tc", flops, "s2e_tapconv_wgrad", _desc(B, Hi, Wi, Cin, Hi, Wi, 64, one, L.ACT_NONE), L.ptr(x), L.ptr(G), L.ptr(dwp),
                        L.IMPL_TC, st, tag="wgrad-head B%d %dx%d Cin%d Cout64 T1" % (B, Hi, Wi, Cin))
            gw = dwp[:len(taps)].t().reshape(weight.shape).contiguous()
        if need_b:
            gb = dy.float().sum().reshape(1)
        return dx, None, gw, gb


def head_conv(x, cfg, weight, bias=None):
    """-> logits (B, Ho, Wo, 1) bf16.  For an even batch the tensor carries `_s2e_gan_sums` (6 floats: per half of the batch
    sum y, sum min(y-1, 0), sum min(-y-1, 0)), which GANLoss picks up instead of reducing the logits again."""
    y, sums = HeadConvFn.apply(x, cfg, weight, bias)
    if sums is not None:
        y._s2e_gan_sums = sums
    return y


def gan_presummed(pred, kind, coef):
    """coef * sum f(pred) for f = identity / hinge-real / hinge-fake when `pred` is one half of a logit tensor whose gather
    kernel already reduced it (pix2pix_model.divide_pred tags the halves); None otherwise."""
    tag = getattr(pred, '_s2e_gan_half', None)
    col = {L.RED_SUM: 0, L.RED_HINGE_REAL: 1, L.RED_HINGE_FAKE: 2}.get(kind)
    if tag is None or col is None:
        return None
    sums, half, version = tag
    if pred._version != version or not pred.is_contiguous():
        return None
    _state["gan_presummed"] = _state.get("gan_presummed", 0) + 1
    return PrecomputedLossFn.apply(pred, None, sums, 3 * half + col, kind, coef)


def _sn_scratch_floats(rows, cols):
    return rows + cols + ((rows + 63) // 64) * cols


def spectral_batch(layers, training, n_calls=1, keep_uv=False):
    """Power iteration for a list of independent spectral-normed layers [(weight_orig, u, v), ...] in four launches per
    iteration (s2e_spectral_power_iter_multi) instead of four per layer.  torch.nn.utils.spectral_norm semantics
    (reference normalization.py:26, architecture.py:31-34): in training mode u and v advance in place, once per call.

    n_calls > 1 reproduces n_calls successive forward calls of every layer (the reference runs netE once per sample,
    pix2pix_model.py:285).  Returns per layer: inv (n_calls,) = 1/sigma of each call and, with keep_uv, the (u, v) each
    call used as U (n_calls, rows), V (n_calls, cols) -- needed by the chain rule of the batched style encoder."""
    if not layers:
        return []
    dev = layers[0][0].device
    dims = [(w.shape[0], w.numel() // w.shape[0]) for w, _, _ in layers]
    inv_all = torch.empty(len(layers) * n_calls, dtype=F32, device=dev)
    scratch = torch.empty(sum(_sn_scratch_floats(r, c) for r, c in dims), dtype=F32, device=dev)
    jobs, out, soff = [], [], 0
    for i, ((w, u, v), (rows, cols)) in enumerate(zip(layers, dims)):
        inv = inv_all[i * n_calls:(i + 1) * n_calls]
        U = V = None
        if keep_uv:
            U = torch.empty(n_calls, rows, dtype=F32, device=dev)
            V = torch.empty(n_calls, cols, dtype=F32, device=dev)
        j = L.SnJob()
        j.w, j.u, j.v, j.inv_sigma = w.detach().data_ptr(), u.data_ptr(), v.data_ptr(), inv.data_ptr()
        j.scratch = scratch.data_ptr() + 4 * soff
        j.u_copy = U.data_ptr() if (keep_uv and training) else None
        j.v_copy = V.data_ptr() if (keep_uv and training) else None
        j.rows, j.cols = rows, cols
        soff += _sn_scratch_floats(rows, cols)
        jobs.append(j)
        out.append((inv, U, V))
    arr = (L.SnJob * len(jobs))(*jobs)
    L.call("s2e_spectral_power_iter_multi", arr, len(jobs), 1 if training else 0, n_calls if training else 1, L.stream())
    if not training:
        for (inv, U, V), (w, u, v) in zip(out, layers):
            if n_calls > 1:
                inv.copy_(inv[:1].expand_as(inv))
            if keep_uv:
                U.copy_(u.expand_as(U))
                V.copy_(v.expand_as(V))
    return out


def spectral_inv_sigma(weight_orig, u, v, training):
    """One power iteration in place on (u, v) (training mode) and 1/sigma as a device scalar."""
    return spectral_batch([(weight_orig, u, v)], training)[0][0]


def spectral_multi(weight_orig, u, v, training, n_calls):
    """What `n_calls` successive forward calls of one spectral-normed layer do to (u, v): (inv, U, V)."""
    return spectral_batch([(weight_orig, u, v)], training, n_calls, keep_uv=True)[0]


def prepare_spectral(convs, training, n_calls=1, keep_uv=False):
    """Run the power iteration of every spectral-normed layer of a network up front, in one batched call, and park
    the results on the layers (`_sn_ready`); each layer's next forward consumes its entry instead of launching its own
    iteration.  The layers are independent, so this is observationally identical to iterating at the point of use."""
    convs = [c for c in convs if getattr(c, 'spectral', False)]
    res = spectral_batch([(c.weight_orig, c.weight_u, c.weight_v) for c in convs], training, n_calls, keep_uv)
    for c, r in zip(convs, res):
        c._sn_ready = r


# ------------------------------------------------------------------------------------------------ norms
# sync: BatchNorm statistics shared by all ranks of the default process group (SyncBatchNorm, `spadesyncbatch`)
NormCfg = namedtuple("NormCfg", "per_sample act training momentum eps sync", defaults=(False,))


_stats_memo = {"ref": None, "key": None, "acc": None}


def clear_stats_memo():
    _stats_memo["ref"] = _stats_memo["key"] = _stats_memo["acc"] = None


def synced(cfg):
    """Whether a normalisation with this config takes the statistics of the global batch over several ranks: BatchNorm
    statistics in training mode under a process group of more than one rank.  Every rank must then run the same
    training-mode forwards (and their backwards) in the same order -- each one issues a collective, as with
    torch.nn.SyncBatchNorm -- on the default (NCCL) group, interleaved with the gradient all-reduces."""
    return cfg.sync and cfg.training and not cfg.per_sample and parallel.world_size() > 1


def _merged_record(x):
    """acc and element count (device, fp64) of x's statistics over the global batch: every rank's s2e_norm_stats record and
    count are all-gathered, then combined by s2e_norm_merge."""
    B, Hx, Wx, Cc = x.shape
    st = L.stream()
    rec = torch.empty(3 * Cc + 1, dtype=torch.float64, device=x.device)
    L.call("s2e_norm_stats", L.ptr(x), B, Hx * Wx, Cc, 0, L.ptr(rec), st)
    rec[3 * Cc:].fill_(float(B * Hx * Wx))      # elements summed (the source's, when x is up-sampled)
    world = parallel.world_size()
    recs = torch.empty(world * (3 * Cc + 1), dtype=torch.float64, device=x.device)
    torch.distributed.all_gather_into_tensor(recs, rec)
    acc = torch.empty(3 * Cc, dtype=torch.float64, device=x.device)
    count = torch.empty(1, dtype=torch.float64, device=x.device)
    L.call("s2e_norm_merge", L.ptr(recs), world, Cc, L.ptr(acc), L.ptr(count), st)
    return acc, count


def spade_statistics(x, cfg, running_mean, running_var, nbt, up):
    """mean / rstd of the param-free norm of SPADE (normalization.py:73-75,91): batch statistics in training mode (also
    advancing BatchNorm's running buffers exactly like torch does) or for InstanceNorm, running statistics in eval mode.
    up: x is the half-resolution source of the real (nearest-2x up-sampled) input -- same mean and variance."""
    B, Hx, Wx, Cc = x.shape
    H, W = (2 * Hx, 2 * Wx) if up else (Hx, Wx)
    st = L.stream()
    G = B if cfg.per_sample else 1
    batch_stats = cfg.per_sample or cfg.training or running_mean is None
    if not batch_stats:   # BatchNorm2d in eval mode
        return running_mean.detach().clone().view(1, Cc), torch.rsqrt(running_var.detach() + cfg.eps).view(1, Cc), False
    mean = torch.empty(G, Cc, dtype=F32, device=x.device)
    rstd = torch.empty(G, Cc, dtype=F32, device=x.device)
    upd = (not cfg.per_sample) and cfg.training and running_mean is not None
    count = float(H * W if cfg.per_sample else B * H * W)     # elements BatchNorm sees (unbiased running_var)
    count_stats = count / 4 if up else count                  # elements actually summed (the 4x smaller source)
    # norm_s and norm_0 of a block with a learned shortcut normalise the SAME tensor (architecture.py:44-49): the sums are
    # taken once (with shared statistics: merged across ranks once, one collective), each layer finalises them into its
    # own mean / rstd / running buffers
    sync = synced(cfg)
    memo = _stats_memo
    key = (x.data_ptr(), x._version, tuple(x.shape), int(cfg.per_sample), sync)
    if memo["ref"] is not None and memo["ref"]() is not None and memo["key"] == key:   # the summed tensor is still alive: same data
        acc = memo["acc"]
        _state["stats_shared"] = _state.get("stats_shared", 0) + 1
    elif sync:
        acc = _merged_record(x)
        _state["sync_collectives"] = _state.get("sync_collectives", 0) + 1
        memo["ref"], memo["key"], memo["acc"] = _weakref.ref(x), key, acc
    else:
        acc = torch.empty(G * 3 * Cc, dtype=torch.float64, device=x.device)    # [sum (x-p)][sum (x-p)^2][pivot p] per group
        L.call("s2e_norm_stats", L.ptr(x), B, Hx * Wx, Cc, int(cfg.per_sample), L.ptr(acc), st)
        memo["ref"], memo["key"], memo["acc"] = _weakref.ref(x), key, acc
    if sync:
        acc, n = acc
        L.call("s2e_norm_finalize_merged", L.ptr(acc), L.ptr(n), Cc, 4.0 if up else 1.0, cfg.eps, L.ptr(mean), L.ptr(rstd),
               L.ptr(running_mean), L.ptr(running_var), cfg.momentum, L.ptr(nbt), st)
        return mean, rstd, True
    L.call("s2e_norm_finalize", L.ptr(acc), G, Cc, count_stats, count, cfg.eps, L.ptr(mean), L.ptr(rstd),
           L.ptr(running_mean) if upd else None, L.ptr(running_var) if upd else None, cfg.momentum,
           L.ptr(nbt) if upd else None, st)
    return mean, rstd, True


def spade_conv_fused_ok(x, up, n_hidden):
    """Shapes the fused gamma|beta-convolution + modulation kernel takes: C in {64, 128} (gamma | beta = one N tile) and
    maps large enough that a 128-pixel tile never spans two samples."""
    B, Hx, Wx, Cc = x.shape
    H, W = (2 * Hx, 2 * Wx) if up else (Hx, Wx)
    if Cc not in (64, 128) or n_hidden % 64 or _state["force_impl"] == L.IMPL_SIMT:
        return False
    tw, th = _fused_tile(H, W, Cc)  # tile = tw x th pixels inside one image
    tiles = ((W + tw - 1) // tw) * ((H + th - 1) // th)
    return (tw == 8 or H % th == 0) and tiles % 2 == 0


def spade_conv_fused(actv, conv_cfg, weights, biases, x, style, cfg, running_mean, running_var, nbt, up):
    """Inference / no-grad SPADE+Style block: act(0.5*[norm(x)(1+gamma)+beta + x(1+s0)+s1]) with gamma|beta = conv(actv)
    formed in the tcgen05 accumulator and consumed in the epilogue -- gamma|beta never reach HBM (saves 8 of the 12 bytes
    per element that the convolution output + the modulation kernel move).  No autograd graph is built."""
    assert not torch.is_grad_enabled()
    x, actv = _c(x), _c(actv)
    style = _c(style) if style is not None else None      # None: plain SPADE (no style term, no 1/2)
    B, Hx, Wx, Cc = x.shape
    H, W = (2 * Hx, 2 * Wx) if up else (Hx, Wx)
    assert actv.shape[:3] == (B, H, W) and (style is None or style.shape == (B, 2 * Cc))
    mean, rstd, _ = spade_statistics(x, cfg, running_mean, running_var, nbt, up)
    st = L.stream()
    par = torch.empty(B, 4, Cc, dtype=F32, device=x.device)
    L.call("s2e_spade_params", L.ptr(mean), L.ptr(rstd), L.ptr(style), B, Cc, int(cfg.per_sample), L.ptr(par), st)
    wp = packed_weights(weights, conv_cfg, False)
    bias = torch.cat([b.detach() for b in biases])
    taps = conv_taps(conv_cfg)
    tw, th = _fused_tile(H, W, Cc)
    d = _desc(B, H, W, actv.shape[3], H, W, 2 * Cc, taps, L.ACT_NONE)
    d.tile_w, d.tile_h, d.tile_b = tw, th, 1
    d.spade_x, d.spade_par, d.spade_C, d.spade_act, d.spade_up = L.ptr(x), L.ptr(par), Cc, cfg.act, int(up)
    d.spade_plain = int(style is None)
    out = torch.empty(B, H, W, Cc, dtype=BF16, device=x.device)
    flops = 2.0 * B * H * W * 2 * Cc * weights[0].shape[1] * conv_cfg.kh * conv_cfg.kw
    _timed_call("tc", flops, "s2e_tapconv_fwd", d, L.ptr(actv), L.ptr(wp), L.ptr(bias), None, L.ptr(out), L.IMPL_TC, st,
                tag="fwd+spade B%d %dx%d Cin%d Cout%d T%d" % (B, H, W, actv.shape[3], 2 * Cc, len(taps)))
    return out


class GradSink:
    """Shared gradient buffer of the SpadeStyleFn calls that consume the SAME input x (norm_0 and norm_s of a ResNet
    block with a learned shortcut): the first backward to run allocates the buffer, the others add into it in place
    (dx_accumulate), and only the LAST one hands the gradient to autograd, so no separate add over the (large)
    gradient is ever launched.  Every registered user must take part in the backward pass (true for the block: both
    branches reach the output)."""
    __slots__ = ("buf", "users", "seen")

    def __init__(self):
        self.buf, self.users, self.seen = None, 0, 0


def _spade_style_bwd(synced, dout, amask, x, gb, style, mean, rstd, B, HW, Cc, stat_mode, act, dx, accumulate, dgb, dstyle, chsum,
                     up_w, gb_stride, tag):
    """s2e_spade_style_bwd; with statistics shared across ranks (`synced`), its two halves with the all-reduce of the
    per-channel sums S1, S2 and of the element count between them, so that dx is the gradient of the global-batch
    normalisation.  The 1/world_size factor that the multi-rank graph step puts on the loss is the same on every rank: it
    scales every rank's S1, S2 alike, and S / (global count) stays consistent with the loss that is differentiated."""
    st = L.stream()
    # double [B][5][C], float m12 [B][2][C], then the batch-statistics sums double [2][C] + 1
    racc = torch.empty(B * 5 * Cc + B * Cc + 2 * Cc + 1, dtype=torch.float64, device=x.device)
    args = (L.ptr(dout), L.ptr(amask), L.ptr(x), L.ptr(gb), L.ptr(style), L.ptr(mean), L.ptr(rstd), B, HW, Cc, stat_mode, act,
            L.ptr(racc))
    if not synced:
        _timed_call("normb", 12.0 * B * HW * Cc, "s2e_spade_style_bwd", *args, L.ptr(dx), int(accumulate), L.ptr(dgb),
                    L.ptr(dstyle), L.ptr(chsum), up_w, gb_stride, st, tag=tag)
        return
    sums = racc[B * 6 * Cc:]
    _timed_call("normb", 4.0 * B * HW * Cc, "s2e_spade_style_bwd_reduce", *args, L.ptr(sums), L.ptr(dstyle), L.ptr(chsum),
                up_w, gb_stride, st, tag=tag + " reduce")
    torch.distributed.all_reduce(sums)
    _state["sync_collectives"] = _state.get("sync_collectives", 0) + 1
    _timed_call("normb", 8.0 * B * HW * Cc, "s2e_spade_style_bwd_apply", *args, L.ptr(sums), L.ptr(dx), int(accumulate),
                L.ptr(dgb), up_w, gb_stride, st, tag=tag + " apply")


class SpadeStyleFn(torch.autograd.Function):
    """out = act(0.5 * [ norm(x) * (1 + gamma) + beta + x * (1 + s0) + s1 ])  (normalization.py:91-105,161-192).

    up=True: x is the (B, H/2, W/2, C) tensor whose nearest-2x up-sampling (generator.py:50,86-93) is the block input; gb
    and the output live at (H, W).  The up-sampled copy is never written: the kernels read x through an index map, the
    batch statistics of x and of its up-sampling are identical, and backward reduces the (H, W) gradient 2x2."""

    @staticmethod
    def forward(ctx, x, gb, style, cfg, running_mean, running_var, nbt, up=False, sink=None):
        ctx.sink, ctx.up = sink, up
        if sink is not None:
            sink.users += 1
        x, gb = _c(x), _c(gb)
        style = _c(style) if style is not None else None      # None: plain SPADE, out = act(norm(x)(1+gamma)+beta)
        B, Hx, Wx, Cc = x.shape
        H, W = (2 * Hx, 2 * Wx) if up else (Hx, Wx)
        assert gb.shape == (B, H, W, 2 * Cc) and (style is None or (style.shape == (B, 2 * Cc) and style.dtype == F32))
        st = L.stream()
        mean, rstd, batch_stats = spade_statistics(x, cfg, running_mean, running_var, nbt, up)
        out = torch.empty(B, H, W, Cc, dtype=BF16, device=x.device)
        # backward needs only the sign of `out` (LeakyReLU mask): one bit per element, written by the forward kernel
        amask = None
        ctx.plain = style is None
        if cfg.act != L.ACT_NONE and any(ctx.needs_input_grad[:3]):
            amask = torch.empty(B * H * W * (Cc // 8), dtype=torch.uint8, device=x.device)
        _timed_call("norm", 8.0 * B * H * W * Cc, "s2e_spade_style_fwd", L.ptr(x), L.ptr(gb), L.ptr(style), L.ptr(mean),
                    L.ptr(rstd), B, H * W, Cc, int(cfg.per_sample), cfg.act, L.ptr(out), L.ptr(amask), W if up else 0, st,
                    tag="B%d HW%d C%d%s" % (B, H * W, Cc, " up" if up else ""))
        ctx.cfg, ctx.batch_stats, ctx.hw, ctx.synced = cfg, batch_stats, (H, W), synced(cfg)
        ctx.save_for_backward(x, gb, style, mean, rstd, amask)
        return out

    @staticmethod
    def backward(ctx, dout):
        cfg, up, sink = ctx.cfg, ctx.up, ctx.sink
        x, gb, style, mean, rstd, amask = ctx.saved_tensors
        dout = _c(dout)
        B, Cc = x.shape[0], x.shape[3]
        H, W = ctx.hw
        accumulate = sink is not None and sink.buf is not None
        # gradient w.r.t. x itself: with `up` the kernel adds the four output pixels of every source pixel on the spot (the
        # adjoint of the nearest-2x up-sampling), so the full-resolution gradient is never written
        dx = sink.buf if accumulate else torch.empty_like(x)
        last = True
        if sink is not None:
            sink.seen += 1
            last = sink.seen == sink.users
            sink.buf = None if last else dx       # no reference outlives the backward pass
            if last:
                sink.seen = 0
        dgb = torch.empty_like(gb)
        dstyle = torch.empty_like(style) if style is not None else None
        chsum = torch.empty(3 * Cc, dtype=F32, device=x.device)
        # eval-mode BatchNorm (running statistics): the statistics are constants, bit 1 of the per_sample argument says so
        stat_mode = int(cfg.per_sample) | (0 if ctx.batch_stats else 2)
        _spade_style_bwd(ctx.synced, dout, amask, x, gb, style, mean, rstd, B, H * W, Cc, stat_mode, cfg.act, dx, accumulate, dgb,
                         dstyle, chsum, W if up else 0, 0, "bwd B%d HW%d C%d%s" % (B, H * W, Cc, " up" if up else ""))
        # per-channel sums of the two gradients, for the bias gradients of the convolutions that receive them as dy
        # (TapConvFn.backward picks the attribute up when the tensor reaches it unmodified; otherwise it sums itself)
        dgb._s2e_chsum, dgb._s2e_chsum_ver = chsum[:2 * Cc], (dgb._version, dgb.data_ptr())
        gx = None
        if last:
            gx = dx
            if sink is None and not up and ctx.batch_stats:
                gx._s2e_chsum, gx._s2e_chsum_ver = chsum[2 * Cc:], (gx._version, gx.data_ptr())
        return gx, dgb, dstyle, None, None, None, None, None, None


def _fused_tile_w(W):
    tw = min(W, 128)
    while W % tw or 128 % tw:
        tw -= 1
    return tw


def _fused_tile(H, W, Cc):
    """(tile_w, tile_h) of the fused gamma|beta + modulation kernel: 8 x 16 when the halo-tile kernel applies (N = 2C = 128
    only), else the widest row tile."""
    if Cc == 64 and halo_on() and W >= 8 and H >= 16 and (((W + 7) // 8) * ((H + 15) // 16)) % 2 == 0:
        return 8, 16
    tw = _fused_tile_w(W)
    return tw, 128 // tw


class SpadeConvFn(torch.autograd.Function):
    """Training-mode SPADE+Style block with the gamma|beta convolution and the modulation in ONE tcgen05 kernel
    (normalization.py:85-105,161-192):

        gamma|beta = conv3x3(actv, W_gamma|W_beta) + b      (accumulator only)
        out        = act(0.5 * [ norm(x) * (1 + gamma) + beta + x * (1 + s0) + s1 ])

    The kernel writes `out`, gamma alone (backward needs it; beta is never needed again) and the 1-bit activation mask:
    6 bytes per element instead of the 12 that the convolution output plus the modulation kernel move.  Backward = the
    SPADE+Style backward kernels (dx, dgamma|dbeta, dstyle, bias sums) followed by the convolution's data / weight
    gradients.  Shapes: see spade_conv_fused_ok.  `up` / `sink` as in SpadeStyleFn."""

    @staticmethod
    def forward(ctx, actv, x, style, wg, wb, bg, bb, conv_cfg, cfg, running_mean, running_var, nbt, up, sink):
        ctx.sink, ctx.up = sink, up
        if sink is not None:
            sink.users += 1
        actv, x = _c(actv), _c(x)
        style = _c(style) if style is not None else None      # None: plain SPADE
        B, Hx, Wx, Cc = x.shape
        H, W = (2 * Hx, 2 * Wx) if up else (Hx, Wx)
        Ca = actv.shape[3]
        assert actv.shape == (B, H, W, Ca) and (style is None or style.shape == (B, 2 * Cc)) and cfg.training
        mean, rstd, _ = spade_statistics(x, cfg, running_mean, running_var, nbt, up)
        st = L.stream()
        par = torch.empty(B, 4, Cc, dtype=F32, device=x.device)
        L.call("s2e_spade_params", L.ptr(mean), L.ptr(rstd), L.ptr(style), B, Cc, int(cfg.per_sample), L.ptr(par), st)
        weights = (wg, wb)
        wp = packed_weights(weights, conv_cfg, False)
        bias = torch.cat([bg.detach(), bb.detach()])
        taps = conv_taps(conv_cfg)
        out = torch.empty(B, H, W, Cc, dtype=BF16, device=x.device)
        gamma = torch.empty(B, H, W, Cc, dtype=BF16, device=x.device)
        amask = torch.empty(B * H * W * (Cc // 8), dtype=torch.uint8, device=x.device) if cfg.act != L.ACT_NONE else None
        d = _desc(B, H, W, Ca, H, W, 2 * Cc, taps, L.ACT_NONE)
        tw, th = _fused_tile(H, W, Cc)
        d.tile_w, d.tile_h, d.tile_b = tw, th, 1
        d.spade_x, d.spade_par, d.spade_C, d.spade_act, d.spade_up = L.ptr(x), L.ptr(par), Cc, cfg.act, int(up)
        d.spade_plain = int(style is None)
        d.spade_gamma_out, d.spade_mask_out = L.ptr(gamma), L.ptr(amask)
        flops = 2.0 * B * H * W * 2 * Cc * Ca * conv_cfg.kh * conv_cfg.kw
        _timed_call("tc", flops, "s2e_tapconv_fwd", d, L.ptr(actv), L.ptr(wp), L.ptr(bias), None, L.ptr(out), L.IMPL_TC, st,
                    tag="fwd+spade B%d %dx%d Cin%d Cout%d T%d" % (B, H, W, Ca, 2 * Cc, len(taps)))
        ctx.cfg, ctx.conv_cfg, ctx.hw, ctx.flops, ctx.synced = cfg, conv_cfg, (H, W), flops, synced(cfg)
        ctx.skip_wgrad = _state["skip_wgrad"]
        ctx.weights = weights
        ctx.save_for_backward(actv, x, gamma, style, mean, rstd, amask)
        return out

    @staticmethod
    def backward(ctx, dout):
        cfg, ccfg, up, sink = ctx.cfg, ctx.conv_cfg, ctx.up, ctx.sink
        actv, x, gamma, style, mean, rstd, amask = ctx.saved_tensors
        wg, wb = ctx.weights
        dout = _c(dout)
        B, Cc = x.shape[0], x.shape[3]
        H, W = ctx.hw
        Ca = actv.shape[3]
        st = L.stream()
        # ---- SPADE+Style backward (gamma kept alone: stride Cc)
        accumulate = sink is not None and sink.buf is not None
        dx = sink.buf if accumulate else torch.empty_like(x)      # at x's own resolution (see SpadeStyleFn.backward)
        last = True
        if sink is not None:
            sink.seen += 1
            last = sink.seen == sink.users
            sink.buf = None if last else dx
            if last:
                sink.seen = 0
        dgb = torch.empty(B, H, W, 2 * Cc, dtype=BF16, device=x.device)
        dstyle = torch.empty_like(style) if style is not None else None
        chsum = torch.empty(3 * Cc, dtype=F32, device=x.device)
        _spade_style_bwd(ctx.synced, dout, amask, x, gamma, style, mean, rstd, B, H * W, Cc, int(cfg.per_sample), cfg.act, dx,
                         accumulate, dgb, dstyle, chsum, W if up else 0, Cc, "bwd B%d HW%d C%d%s" % (B, H * W, Cc, " up" if up else ""))
        gx = None
        if last and ctx.needs_input_grad[1]:
            gx = dx
            if sink is None and not up:     # bias gradient of the convolution that produced x (see SpadeStyleFn)
                gx._s2e_chsum, gx._s2e_chsum_ver = chsum[2 * Cc:], (gx._version, gx.data_ptr())
        # ---- gamma|beta convolution backward
        taps = conv_taps(ccfg)
        dactv = None
        if ctx.needs_input_grad[0]:
            wpt = packed_weights((wg, wb), ccfg, True)
            dd = _desc(B, H, W, 2 * Cc, H, W, Ca, taps, L.ACT_NONE, negate=True)
            if ccfg.relu_in:
                dd.relu_mask = L.ptr(actv)   # actv = relu(.) > 0 exactly where the ReLU passed gradient
            dactv = torch.empty_like(actv)
            _timed_call("tc", ctx.flops, "s2e_tapconv_fwd", dd, L.ptr(dgb), L.ptr(wpt), None, None, L.ptr(dactv), L.IMPL_TC, st,
                        tag="dgrad B%d %dx%d Cin%d Cout%d T%d" % (B, H, W, 2 * Cc, Ca, len(taps)))
        gwg = gwb = gbg = gbb = None
        if not ctx.skip_wgrad:
            if ctx.needs_input_grad[3] or ctx.needs_input_grad[4]:
                dwp = torch.zeros(len(taps) * 2 * Cc * Ca, dtype=F32, device=x.device)
                d = _desc(B, H, W, Ca, H, W, 2 * Cc, taps, L.ACT_NONE)
                _timed_call("tc", ctx.flops, "s2e_tapconv_wgrad", d, L.ptr(actv), L.ptr(dgb), L.ptr(dwp), L.IMPL_TC, st,
                            tag="wgrad B%d %dx%d Cin%d Cout%d T%d" % (B, H, W, Ca, 2 * Cc, len(taps)))
                outs = []
                for i, w in enumerate((wg, wb)):
                    g = torch.empty_like(w)
                    L.call("s2e_unpack_wgrad", L.ptr(dwp), Cc, Ca, ccfg.kh, ccfg.kw, 1, ccfg.pad, 2 * Cc, i * Cc, 0,
                           L.ptr(w.detach()), None, None, None, None, L.ptr(g), 0, st)
                    outs.append(g)
                gwg, gwb = outs
            if ctx.needs_input_grad[5] or ctx.needs_input_grad[6]:
                gbg, gbb = chsum[:Cc].clone(), chsum[Cc:2 * Cc].clone()   # sum dgamma, sum dbeta: free from the reduce pass
                _state["chsum_hits"] = _state.get("chsum_hits", 0) + 1
        return dactv, gx, dstyle, gwg, gwb, gbg, gbb, None, None, None, None, None, None, None


class InstNormFn(torch.autograd.Function):
    """nn.InstanceNorm2d(affine=False, eps=1e-5) + optional LeakyReLU(0.2) on NHWC bf16.

    With `sn = (inv_sigma (S,), U (S,Cout), V (S,K), group, weight_orig)` the input is the UNSCALED output z of a
    spectral-normed convolution applied to S groups of `group` images; group s is normalised as IN(z / sigma_s)
    (the scale only enters the statistics) and backward additionally returns, as the gradient of `weight_orig`, the
    spectral chain-rule term  - sum_s c_s u_s v_s^T  (see s2e_sn_in_correction)."""

    @staticmethod
    def forward(ctx, x, act, sn_inv=None, sn_U=None, sn_V=None, group=1, weight_orig=None, pair_l1=None):
        """pair_l1 (optional, one zeroed float): x holds the [fake ; real] halves of a discriminator feature; the kernel adds
        sum |y[:B/2] - y[B/2:]| to it (the feature-matching reduction rides in the apply pass)."""
        x = _c(x)
        B, H, W, Cc = x.shape
        acc = torch.empty(B * 3 * Cc, dtype=torch.float64, device=x.device)
        mean = torch.empty(B, Cc, dtype=F32, device=x.device)
        rstd = torch.empty(B, Cc, dtype=F32, device=x.device)
        y = torch.empty_like(x)
        L.call("s2e_instnorm_fwd", L.ptr(x), B, H * W, Cc, act, 1e-5, L.ptr(sn_inv), group, L.ptr(acc), L.ptr(mean),
               L.ptr(rstd), L.ptr(y), L.ptr(pair_l1), L.stream())
        ctx.act, ctx.group = act, group
        ctx.skip_wgrad = _state["skip_wgrad"]    # captured at forward time, like TapConvFn
        ctx.has_sn = sn_inv is not None
        ctx.save_for_backward(x, mean, rstd, sn_inv, sn_U, sn_V, weight_orig)   # not y: backward takes the activation's sign from x
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mean, rstd, sn_inv, sn_U, sn_V, weight_orig = ctx.saved_tensors
        dy = _c(dy)
        B, H, W, Cc = x.shape
        racc = torch.empty(B * 2 * Cc, dtype=torch.float64, device=x.device)
        dx = torch.empty_like(x)
        st = L.stream()
        L.call("s2e_instnorm_bwd", L.ptr(dy), None, L.ptr(x), L.ptr(mean), L.ptr(rstd), B, H * W, Cc, ctx.act,
               L.ptr(racc), L.ptr(dx), st)
        gw = None
        if ctx.has_sn and weight_orig is not None and ctx.needs_input_grad[6] and not ctx.skip_wgrad:
            S = sn_inv.shape[0]
            K = weight_orig.numel() // weight_orig.shape[0]
            coef = torch.empty(S, dtype=F32, device=x.device)
            gw = torch.empty_like(weight_orig)
            L.call("s2e_sn_in_correction", L.ptr(racc), L.ptr(rstd), L.ptr(sn_inv), S, ctx.group, Cc, 1e-5, L.ptr(sn_U),
                   L.ptr(sn_V), K, L.ptr(coef), L.ptr(gw), st)
        return dx, None, None, None, None, None, gw, None


@contextlib.contextmanager
def fm_pair_sums():
    """While active, InstanceNorm layers fed with an even batch also reduce sum |y[:B/2] - y[B/2:]| (layers.InstanceNorm2d): the
    generator step's discriminator pass, whose features enter the feature-matching loss."""
    prev = _state.get("fm_pairs", False)
    _state["fm_pairs"] = True
    try:
        yield
    finally:
        _state["fm_pairs"] = prev


@contextlib.contextmanager
def head_sign_sums():
    """While active, head_conv on an even ([fake ; real]) batch also sums sign(y) over the real half, in the gather kernel
    that produces the logits (s2e_head_gather_signs).  Yields {logits data_ptr: (1,) fp32 sum} of those launches: the
    discriminator step's statistic for --ada_target."""
    prev = _state.get("sign_sums")
    _state["sign_sums"] = found = {}
    try:
        yield found
    finally:
        _state["sign_sums"] = prev


# ------------------------------------------------------------------------------------------------ elementwise / resampling
class Upsample2xFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        B, H, W, Cc = x.shape
        y = torch.empty(B, 2 * H, 2 * W, Cc, dtype=BF16, device=x.device)
        L.call("s2e_upsample2x_fwd", L.ptr(x), B, H, W, Cc, L.ptr(y), L.stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _c(dy)
        B, H2, W2, Cc = dy.shape
        dx = torch.empty(B, H2 // 2, W2 // 2, Cc, dtype=BF16, device=dy.device)
        L.call("s2e_upsample2x_bwd", L.ptr(dy), B, H2 // 2, W2 // 2, Cc, L.ptr(dx), L.stream())
        return dx


class AddFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        a, b = _c(a), _c(b)
        y = torch.empty_like(a)
        L.call("s2e_add", L.ptr(a), L.ptr(b), a.numel(), L.ptr(y), L.stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        return dy, dy


class ActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, act):
        x = _c(x)
        y = torch.empty_like(x)
        L.call("s2e_act_fwd", L.ptr(x), x.numel(), act, L.ptr(y), L.stream())
        ctx.act = act
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = _c(dy)
        dx = torch.empty_like(dy)
        L.call("s2e_act_bwd", L.ptr(dy), L.ptr(y), dy.numel(), ctx.act, L.ptr(dx), L.stream())
        return dx, None


class AvgPool3s2Fn(torch.autograd.Function):
    """F.avg_pool2d(k=3, s=2, p=1, count_include_pad=False) (discriminator.py:46-49)."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        B, H, W, Cc = x.shape
        y = torch.empty(B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, Cc, dtype=BF16, device=x.device)
        L.call("s2e_avgpool3s2_fwd", L.ptr(x), B, H, W, Cc, L.ptr(y), L.stream())
        ctx.shape = (B, H, W, Cc)
        return y

    @staticmethod
    def backward(ctx, dy):
        B, H, W, Cc = ctx.shape
        dy = _c(dy)
        dx = torch.empty(B, H, W, Cc, dtype=BF16, device=dy.device)
        L.call("s2e_avgpool3s2_bwd", L.ptr(dy), B, H, W, Cc, L.ptr(dx), L.stream())
        return dx


class BilinearFn(torch.autograd.Function):
    """F.interpolate(x, size, mode='bilinear', align_corners=False) of (N,1,H,W) fp32 -> (N,Hd,Wd,1) bf16."""

    @staticmethod
    def forward(ctx, x, size):
        x = _c(x.float())
        N, Cc, Hs, Ws = x.shape
        y = torch.empty(N * Cc, size[0], size[1], 1, dtype=BF16, device=x.device)
        L.call("s2e_bilinear_fwd", L.ptr(x), N * Cc, Hs, Ws, size[0], size[1], L.ptr(y), L.stream())
        ctx.shape, ctx.size = (N, Cc, Hs, Ws), size
        return y

    @staticmethod
    def backward(ctx, dy):
        N, Cc, Hs, Ws = ctx.shape
        dy = _c(dy)
        dx = torch.empty(N, Cc, Hs, Ws, dtype=F32, device=dy.device)
        L.call("s2e_bilinear_bwd", L.ptr(dy), N * Cc, Hs, Ws, ctx.size[0], ctx.size[1], L.ptr(dx), L.stream())
        return dx, None


class ToNHWCFn(torch.autograd.Function):
    """(B,C,H,W) fp32 -> (B,H,W,C) bf16."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x.float())
        B, Cc, H, W = x.shape
        y = torch.empty(B, H, W, Cc, dtype=BF16, device=x.device)
        L.call("s2e_nchw_f32_to_nhwc_bf16", L.ptr(x), B, Cc, H, W, L.ptr(y), L.stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _c(dy)
        B, H, W, Cc = dy.shape
        dx = torch.empty(B, Cc, H, W, dtype=F32, device=dy.device)
        L.call("s2e_nhwc_bf16_to_nchw_f32", L.ptr(dy), B, Cc, H, W, L.ptr(dx), L.stream())
        return dx


class ToNCHWFn(torch.autograd.Function):
    """(B,H,W,C) bf16 -> (B,C,H,W) fp32."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        B, H, W, Cc = x.shape
        y = torch.empty(B, Cc, H, W, dtype=F32, device=x.device)
        L.call("s2e_nhwc_bf16_to_nchw_f32", L.ptr(x), B, Cc, H, W, L.ptr(y), L.stream())
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _c(dy.float())
        B, Cc, H, W = dy.shape
        dx = torch.empty(B, H, W, Cc, dtype=BF16, device=dy.device)
        L.call("s2e_nchw_f32_to_nhwc_bf16", L.ptr(dy), B, Cc, H, W, L.ptr(dx), L.stream())
        return dx


def as_nhwc(x):
    """Accept the reference's logical-NCHW tensors.  Our own activations (bf16, NHWC storage seen through a
    permuted view) pass through for free; anything else is converted by the layout kernel."""
    if x.dtype == BF16:
        v = x.permute(0, 2, 3, 1)
        if v.is_contiguous():
            return v
        return ToNHWCFn.apply(x)
    return ToNHWCFn.apply(x)


def as_nchw_view(y):
    return y.permute(0, 3, 1, 2)


def one_hot(label, nc):
    """pix2pix_model.py:144-152 -- (B,1,H,W) integer labels -> (B,nc,H,W) fp32 one-hot (bit-exact)."""
    label = _c(label.long())
    B, _, H, W = label.shape
    out = torch.empty(B, nc, H, W, dtype=F32, device=label.device)
    L.call("s2e_onehot_nchw", L.ptr(label), B, H, W, nc, L.ptr(out), L.stream())
    return out


def seg_nearest(seg, hd, wd, cpad=0):
    """F.interpolate(seg, size, mode='nearest') fused with the NCHW fp32 -> NHWC bf16 layout change.
    cpad > C: the output carries cpad channels, the extra ones zero (a 35-class map padded to 64 channels runs mlp_shared /
    G.fc as ordinary 64-channel tap convolutions on the tensor cores)."""
    seg = _c(seg.detach().float())
    B, Cc, Hs, Ws = seg.shape
    cp = max(cpad, Cc)
    out = torch.empty(B, hd, wd, cp, dtype=BF16, device=seg.device)
    L.call("s2e_seg_nearest_nhwc", L.ptr(seg), B, Cc, Hs, Ws, hd, wd, cp, L.ptr(out), L.stream())
    return out


def seg_im2col(seg, hd, wd):
    """Nearest-resize + 3x3 im2col of the segmap to (B,hd,wd,64) bf16 (see s2e_seg_im2col3x3)."""
    seg = _c(seg.detach().float())
    B, Cc, Hs, Ws = seg.shape
    out = torch.empty(B, hd, wd, 64, dtype=BF16, device=seg.device)
    L.call("s2e_seg_im2col3x3", L.ptr(seg), B, Cc, Hs, Ws, hd, wd, L.ptr(out), L.stream())
    return out


class SegConvFn(torch.autograd.Function):
    """act(conv3x3(seg, W) + b) for a thin segmap given as its 64-channel im2col: one K=64 GEMM on the tcgen05
    kernels, forward and weight gradient (the segmap itself needs no gradient)."""

    @staticmethod
    def forward(ctx, col, weight, bias, act, act_grad_fused=False):
        ctx.act_grad_fused = act_grad_fused   # the consumer already applied the ReLU mask to the gradient it sends back
        B, H, W, K = col.shape
        Cout, Cs = weight.shape[0], weight.shape[1]
        assert K == 64 and weight.shape[2:] == (3, 3) and 9 * Cs <= 62
        wp = packed_weight_im2col(weight, bias)    # the bias rides in column 63 of the GEMM (constant-one channel)
        y = torch.empty(B, H, W, Cout, dtype=BF16, device=col.device)
        d = _desc(B, H, W, 64, H, W, Cout, [(0, 0)], act)
        flops = 2.0 * B * H * W * Cout * Cs * 9
        impl = _pick(Cout % 8 == 0)
        if impl == L.IMPL_TC:
            _timed_call("tc", flops, "s2e_tapconv_fwd", d, L.ptr(col), L.ptr(wp), None, None, L.ptr(y), impl, L.stream(),
                        tag="fwd-seg B%d %dx%d Cin64 Cout%d T1" % (B, H, W, Cout))
        else:
            L.call("s2e_tapconv_fwd", d, L.ptr(col), L.ptr(wp), None, None, L.ptr(y), impl, L.stream())
        ctx.act, ctx.flops, ctx.cs, ctx.has_b = act, flops, Cs, bias is not None
        ctx.skip_wgrad = _state["skip_wgrad"]
        ctx.save_for_backward(col, y, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        col, y, weight = ctx.saved_tensors
        dy = _c(dy)
        B, H, W, Cout = dy.shape
        st = L.stream()
        if ctx.act != L.ACT_NONE and not ctx.act_grad_fused:
            dpre = torch.empty_like(dy)
            L.call("s2e_act_bwd", L.ptr(dy), L.ptr(y), dy.numel(), ctx.act, L.ptr(dpre), st)
        else:
            dpre = dy
        gw = gb = None
        need_b = ctx.has_b and ctx.needs_input_grad[2] and not ctx.skip_wgrad
        if (ctx.needs_input_grad[1] or need_b) and not ctx.skip_wgrad:
            dwp = torch.zeros(Cout * 64, dtype=F32, device=dy.device)
            d = _desc(B, H, W, 64, H, W, Cout, [(0, 0)], L.ACT_NONE)
            impl = _pick(Cout >= 64 and Cout % 8 == 0)
            if impl == L.IMPL_TC:
                _timed_call("tc", ctx.flops, "s2e_tapconv_wgrad", d, L.ptr(col), L.ptr(dpre), L.ptr(dwp), impl, st,
                            tag="wgrad-seg B%d %dx%d Cin64 Cout%d T1" % (B, H, W, Cout))
            else:
                L.call("s2e_tapconv_wgrad", d, L.ptr(col), L.ptr(dpre), L.ptr(dwp), impl, st)
            gw = torch.empty_like(weight)
            gb = torch.empty(Cout, dtype=F32, device=dy.device) if need_b else None   # column 63 = bias gradient
            L.call("s2e_unpack_wgrad_im2col3x3", L.ptr(dwp), Cout, ctx.cs, L.ptr(gw), L.ptr(gb), st)
        return None, gw, gb, None, None


class MakeDInputFn(torch.autograd.Function):
    """cat([cat([seg,fake],1), cat([seg,real],1)], 0) as (2B,H,W,nc+1) bf16 (pix2pix_model.py:328-338)."""

    @staticmethod
    def forward(ctx, seg, fake, real, cpad=0):
        seg, fake, real = _c(seg.float()), _c(fake.float()), _c(real.float())
        B, nc, H, W = seg.shape
        assert fake.shape == (B, 1, H, W) and real.shape == (B, 1, H, W), (fake.shape, real.shape, seg.shape)
        cpad = max(cpad, nc + 1)
        out = torch.empty(2 * B, H, W, cpad, dtype=BF16, device=seg.device)
        L.call("s2e_make_d_input", L.ptr(seg), L.ptr(fake), L.ptr(real), B, nc, H, W, cpad, L.ptr(out), L.stream())
        ctx.dims = (B, nc, H, W)
        ctx.cpad = cpad
        return out

    @staticmethod
    def backward(ctx, dout):
        B, nc, H, W = ctx.dims
        dout = _c(dout)
        dfake = None
        if ctx.needs_input_grad[1]:
            dfake = torch.empty(B, 1, H, W, dtype=F32, device=dout.device)
            L.call("s2e_d_input_grad", L.ptr(dout), B, nc, H, W, ctx.cpad, L.ptr(dfake), L.stream())
        return None, dfake, None, None


DIFFAUG_OPS = (("color", L.DIFFAUG_COLOR), ("xflip", L.DIFFAUG_XFLIP), ("geometric", L.DIFFAUG_GEOMETRIC),
               ("translation", L.DIFFAUG_TRANSLATION), ("cutout", L.DIFFAUG_CUTOUT))
DIFFAUG_GEOM_OPS = L.DIFFAUG_XFLIP | L.DIFFAUG_GEOMETRIC


def parse_diff_augment(policy):
    """'cutout,color' -> ('color', 'cutout'), the bits of the C ABI: the ops always run in the order color -> xflip ->
    geometric -> translation -> cutout, whatever the order of the string.  '' -> ((), 0)."""
    names = [s.strip() for s in (policy or '').split(',') if s.strip()]
    known = dict(DIFFAUG_OPS)
    bad = [n for n in names if n not in known]
    if bad:
        raise ValueError("--diff_augment: unknown op(s) %s (choose from %s)" % (bad, ", ".join(known)))
    ops_ = tuple(n for n, _ in DIFFAUG_OPS if n in names)
    return ops_, sum(known[n] for n in ops_)


def diffaug_draw(state, B, index_offset, H, W):
    """[B, 6] fp32 parameter records (u0, u1, tx, ty, ox, oy) of samples index_offset .. index_offset + B - 1 for an H x W
    map, drawn at the counter in `state` (int64 [seed, counter] on the device), which the launch advances by one."""
    assert state.dtype == torch.int64 and state.numel() == 2 and state.is_contiguous()
    rec = torch.empty(B, L.DIFFAUG_RECORD, dtype=F32, device=state.device)
    L.call("s2e_diffaug_draw", L.ptr(state), B, index_offset, H, W, L.ptr(rec), L.stream())
    return rec


def diffaug_draw_p(state, p, B, index_offset, H, W):
    """diffaug_draw plus the per-op gates at probability `p` (one float64 on the device): -> the [B, 6] records, bit for
    bit diffaug_draw's, and [B] int32 masks of the S2E_DIFFAUG_* bits whose gates passed."""
    assert state.dtype == torch.int64 and state.numel() == 2 and state.is_contiguous()
    assert p.dtype == torch.float64 and p.numel() == 1 and p.device == state.device
    rec = torch.empty(B, L.DIFFAUG_RECORD, dtype=F32, device=state.device)
    mask = torch.empty(B, dtype=torch.int32, device=state.device)
    L.call("s2e_diffaug_draw_p", L.ptr(state), L.ptr(p), B, index_offset, H, W, L.ptr(rec), L.ptr(mask), L.stream())
    return rec, mask


def diffaug_draw_geom(state, p, B, index_offset, H, W):
    """diffaug_draw_p plus the mirror and geometric draws (--diff_augment xflip / geometric): -> the [B, 6] records, bit
    for bit diffaug_draw's, [B, 8] fp32 inverse matrices M (six entries, two zero pads), and [B] int32 masks whose
    COLOR / TRANSLATION / CUTOUT bits are diffaug_draw_p's, plus XFLIP (mirror applied) and GEOMETRIC (a geometric gate
    passed)."""
    assert state.dtype == torch.int64 and state.numel() == 2 and state.is_contiguous()
    assert p.dtype == torch.float64 and p.numel() == 1 and p.device == state.device
    rec = torch.empty(B, L.DIFFAUG_RECORD, dtype=F32, device=state.device)
    geom = torch.empty(B, L.DIFFAUG_GEOM_RECORD, dtype=F32, device=state.device)
    mask = torch.empty(B, dtype=torch.int32, device=state.device)
    L.call("s2e_diffaug_draw_geom", L.ptr(state), L.ptr(p), B, index_offset, H, W, L.ptr(rec), L.ptr(geom), L.ptr(mask),
           L.stream())
    return rec, geom, mask


def _d_input_aug_fwd(ctx, seg, fake, real, cpad, params, policy, opmask, geom=None):
    seg, fake, real = _c(seg.float()), _c(fake.float()), _c(real.float())
    B, nc, H, W = seg.shape
    assert fake.shape == (B, 1, H, W) and real.shape == (B, 1, H, W), (fake.shape, real.shape, seg.shape)
    assert params.shape == (B, L.DIFFAUG_RECORD) and params.dtype == F32 and params.is_contiguous()
    if geom is not None and policy & L.DIFFAUG_GEOMETRIC and (H < 2 or W < 2):
        raise ValueError("--diff_augment geometric needs maps of at least 2 x 2 pixels, got %d x %d" % (H, W))
    cpad = max(cpad, nc + 1)
    st = L.stream()
    means = None
    if policy & L.DIFFAUG_COLOR:
        means = torch.empty(2 * B, dtype=F32, device=seg.device)
        L.call("s2e_diffaug_means", L.ptr(fake), L.ptr(real), B, H, W, L.ptr(means), st)
    out = torch.empty(2 * B, H, W, cpad, dtype=BF16, device=seg.device)
    if geom is not None:
        assert opmask.shape == (B,) and opmask.dtype == torch.int32 and opmask.is_contiguous()
        assert geom.shape == (B, L.DIFFAUG_GEOM_RECORD) and geom.dtype == F32 and geom.is_contiguous()
        L.call("s2e_make_d_input_aug_geom", L.ptr(seg), L.ptr(fake), L.ptr(real), B, nc, H, W, cpad, L.ptr(params),
               L.ptr(means), policy, L.ptr(opmask), L.ptr(geom), L.ptr(out), st)
        ctx.save_for_backward(params, opmask, geom)
    elif opmask is None:
        L.call("s2e_make_d_input_aug", L.ptr(seg), L.ptr(fake), L.ptr(real), B, nc, H, W, cpad, L.ptr(params), L.ptr(means),
               policy, L.ptr(out), st)
        ctx.save_for_backward(params)
    else:
        assert opmask.shape == (B,) and opmask.dtype == torch.int32 and opmask.is_contiguous()
        L.call("s2e_make_d_input_aug_masked", L.ptr(seg), L.ptr(fake), L.ptr(real), B, nc, H, W, cpad, L.ptr(params),
               L.ptr(means), policy, L.ptr(opmask), L.ptr(out), st)
        ctx.save_for_backward(params, opmask)
    ctx.dims = (B, nc, H, W)
    ctx.cpad, ctx.policy = cpad, policy
    return out


def _d_input_aug_bwd(ctx, dout):
    B, nc, H, W = ctx.dims
    dout = _c(dout)
    if not ctx.needs_input_grad[1]:
        return None
    params, *opmask = ctx.saved_tensors       # [], [opmask] or [opmask, geom]
    dfake = torch.empty(B, 1, H, W, dtype=F32, device=dout.device)
    scratch = torch.empty(B, dtype=torch.float64, device=dout.device) if ctx.policy & L.DIFFAUG_COLOR else None
    if not opmask:
        L.call("s2e_d_input_grad_aug", L.ptr(dout), B, nc, H, W, ctx.cpad, L.ptr(params), ctx.policy, L.ptr(scratch),
               L.ptr(dfake), L.stream())
    elif len(opmask) == 2:
        mask, geom = opmask
        L.call("s2e_d_input_grad_aug_geom", L.ptr(dout), B, nc, H, W, ctx.cpad, L.ptr(params), ctx.policy, L.ptr(mask),
               L.ptr(geom), L.ptr(scratch), L.ptr(dfake), L.stream())
    else:
        L.call("s2e_d_input_grad_aug_masked", L.ptr(dout), B, nc, H, W, ctx.cpad, L.ptr(params), ctx.policy, L.ptr(opmask[0]),
               L.ptr(scratch), L.ptr(dfake), L.stream())
    return dfake


class MakeDInputAugFn(torch.autograd.Function):
    """MakeDInputFn with differentiable augmentation (--diff_augment): rows b and B + b use record b of `params`
    (ops.diffaug_draw); colour touches the image channel, translation and cutout every channel."""

    @staticmethod
    def forward(ctx, seg, fake, real, cpad, params, policy):
        return _d_input_aug_fwd(ctx, seg, fake, real, cpad, params, policy, None)

    @staticmethod
    def backward(ctx, dout):
        return None, _d_input_aug_bwd(ctx, dout), None, None, None, None


class MakeDInputAugMaskedFn(torch.autograd.Function):
    """MakeDInputAugFn with per-sample gates (--diff_augment_p, --ada_target): sample b applies policy & opmask[b]
    (ops.diffaug_draw_p)."""

    @staticmethod
    def forward(ctx, seg, fake, real, cpad, params, opmask, policy):
        return _d_input_aug_fwd(ctx, seg, fake, real, cpad, params, policy, opmask)

    @staticmethod
    def backward(ctx, dout):
        return None, _d_input_aug_bwd(ctx, dout), None, None, None, None, None


class MakeDInputAugGeomFn(torch.autograd.Function):
    """MakeDInputAugMaskedFn with the mirror and the geometric warp (--diff_augment xflip / geometric): sample b applies
    policy & opmask[b] and the matrix geom[b] (ops.diffaug_draw_geom).  The labels are sampled at the nearest tap, the
    image bilinearly, both with reflection at the borders; the adjoint is a deterministic gather."""

    @staticmethod
    def forward(ctx, seg, fake, real, cpad, params, opmask, geom, policy):
        return _d_input_aug_fwd(ctx, seg, fake, real, cpad, params, policy, opmask, geom)

    @staticmethod
    def backward(ctx, dout):
        return None, _d_input_aug_bwd(ctx, dout), None, None, None, None, None, None


def ada_update(state, target, kimg, interval):
    """ADA's controller step on `state` (Pix2PixModel.ada_state): adds state['record'] into state['acc'] and, every
    `interval` calls, moves state['p'] (s2e_ada_update)."""
    n_d = (state['record'].numel() - 1) // 2
    L.call("s2e_ada_update", L.ptr(state['record']), n_d, L.ptr(state['acc']), L.ptr(state['pos']), L.ptr(state['p']),
           float(target), float(kimg), int(interval), L.stream())


def sign_sum(x):
    """(1,) fp32 = sum sign(x) of a contiguous tensor (S2E_RED_SIGN; exact below 2^24 elements)."""
    x = _c(x.detach())
    assert x.numel() < 1 << 24
    out = torch.empty(1, dtype=F32, device=x.device)
    L.call("s2e_reduce_loss", L.ptr(x), None, x.numel(), int(x.dtype == F32), L.RED_SIGN, 1.0, 0.0, L.ptr(out), 0, L.stream())
    return out


class TanhFn(torch.autograd.Function):
    """(B,H,W,1) bf16 -> tanh -> (B,1,H,W) fp32 (generator.py:99)."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        B, H, W, Cc = x.shape
        assert Cc == 1
        y = torch.empty(B, 1, H, W, dtype=F32, device=x.device)
        L.call("s2e_tanh_fwd", L.ptr(x), x.numel(), L.ptr(y), L.stream())
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = _c(dy.float())
        B, _, H, W = y.shape
        dx = torch.empty(B, H, W, 1, dtype=BF16, device=y.device)
        L.call("s2e_tanh_bwd", L.ptr(dy), L.ptr(y), y.numel(), L.ptr(dx), L.stream())
        return dx


class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) in fp32.  hw > 0: x is an NHWC bf16 feature (M,h,w,C) flattened in NCHW order with
    LeakyReLU(0.2) applied first (encoder.py:64-68)."""

    @staticmethod
    def forward(ctx, x, w, b, act, hw):
        x = _c(x)
        M = x.shape[0]
        N, K = w.shape
        y = torch.empty(M, N, dtype=F32, device=w.device)
        L.call("s2e_linear_fwd", L.ptr(x), L.ptr(w.detach()), L.ptr(b.detach()) if b is not None else None, M, N, K, act,
               hw, L.ptr(y), L.stream())
        ctx.act, ctx.hw = act, hw
        ctx.save_for_backward(x, w, y)
        ctx.has_b = b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, y = ctx.saved_tensors
        dy = _c(dy.float())
        M, (N, K) = x.shape[0], w.shape
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw = torch.empty_like(w) if ctx.needs_input_grad[1] else None
        db = torch.empty(N, dtype=F32, device=w.device) if (ctx.has_b and ctx.needs_input_grad[2]) else None
        if dw is None and db is not None:
            dw = torch.empty_like(w)
        L.call("s2e_linear_bwd", L.ptr(dy), L.ptr(y), L.ptr(x), L.ptr(w.detach()), M, N, K, ctx.act, ctx.hw, L.ptr(dx),
               L.ptr(dw), L.ptr(db), L.stream())
        return dx, (dw if ctx.needs_input_grad[1] else None), db, None, None


class ReduceLossFn(torch.autograd.Function):
    """(1,) fp32 = coef * sum f(x[, y]) with f selected by `kind` (loss.py:58-83, nn.L1Loss/MSELoss); `target` is the
    constant label of the LS / BCE kinds."""

    @staticmethod
    def forward(ctx, x, y, kind, coef, target=0.0):
        x = _c(x)
        f32 = int(x.dtype == F32)
        if y is not None:
            y = _c(y.detach())
            if y.dtype != x.dtype:
                y = y.to(x.dtype)
            assert y.shape == x.shape
        out = torch.empty(1, dtype=F32, device=x.device)
        L.call("s2e_reduce_loss", L.ptr(x), L.ptr(y), x.numel(), f32, kind, coef, target, L.ptr(out), 0, L.stream())
        ctx.kind, ctx.coef, ctx.f32, ctx.target = kind, coef, f32, target
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, y = ctx.saved_tensors
        gout = _c(gout.float())
        dx = torch.empty_like(x)
        L.call("s2e_reduce_loss_bwd", L.ptr(x), L.ptr(y), x.numel(), ctx.f32, ctx.kind, ctx.coef, ctx.target, L.ptr(gout),
               L.ptr(dx), 0, L.stream())
        return dx, None, None, None, None


def reduce_loss(x, y, kind, coef, target=0.0):
    return ReduceLossFn.apply(x, y, kind, float(coef), float(target))


class HalvesLossFn(torch.autograd.Function):
    """Feature-matching term on a discriminator feature that holds [fake ; real] along the batch axis
    (pix2pix_model.py:233-241): coef * sum f(t[:B] - t[B:]) with the real half detached.  Works on the whole tensor so
    that autograd needs no slice / zero-pad / copy kernels: backward writes the full-size gradient in one pass."""

    @staticmethod
    def forward(ctx, t, kind, coef):
        t = _c(t)
        n2 = t.numel() // 2
        f32 = int(t.dtype == F32)
        out = torch.empty(1, dtype=F32, device=t.device)
        flat = t.view(-1)
        L.call("s2e_reduce_loss", L.ptr(flat), L.ptr(flat[n2:]), n2, f32, kind, coef, 0.0, L.ptr(out), 0, L.stream())
        ctx.kind, ctx.coef, ctx.f32 = kind, coef, f32
        ctx.save_for_backward(t)
        return out

    @staticmethod
    def backward(ctx, gout):
        (t,) = ctx.saved_tensors
        gout = _c(gout.float())
        n2 = t.numel() // 2
        dx = torch.empty_like(t)
        flat, dflat = t.view(-1), dx.view(-1)
        dflat[n2:].zero_()
        L.call("s2e_reduce_loss_bwd", L.ptr(flat), L.ptr(flat[n2:]), n2, ctx.f32, ctx.kind, ctx.coef, 0.0, L.ptr(gout),
               L.ptr(dflat), 0, L.stream())
        return dx, None, None


class HalvesPresummedFn(torch.autograd.Function):
    """HalvesLossFn whose forward reduction was already done by the kernel that produced `t` (InstNormFn with pair_l1):
    coef * pre; backward is HalvesLossFn's."""

    @staticmethod
    def forward(ctx, t, pre, kind, coef):
        ctx.kind, ctx.coef, ctx.f32 = kind, coef, int(t.dtype == F32)
        ctx.save_for_backward(_c(t))
        return pre * coef

    @staticmethod
    def backward(ctx, gout):
        return HalvesLossFn.backward(ctx, gout)[0], None, None, None


class PairLossFn(torch.autograd.Function):
    """coef * sum f(a - b) with gradients to BOTH operands (nn.MSELoss / nn.L1Loss between two live tensors: the style
    losses of pix2pix_model.py:162-184,212-229, whose "real" side is not detached in the reference)."""

    @staticmethod
    def forward(ctx, a, b, kind, coef):
        a, b = _c(a), _c(b)
        assert a.shape == b.shape and a.dtype == b.dtype and a.dtype in (F32, BF16)
        f32 = int(a.dtype == F32)
        out = torch.empty(1, dtype=F32, device=a.device)
        L.call("s2e_reduce_loss", L.ptr(a), L.ptr(b), a.numel(), f32, kind, coef, 0.0, L.ptr(out), 0, L.stream())
        ctx.kind, ctx.coef, ctx.f32 = kind, coef, f32
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    def backward(ctx, gout):
        a, b = ctx.saved_tensors
        gout = _c(gout.float())
        da = db = None
        if ctx.needs_input_grad[0]:
            da = torch.empty_like(a)
            L.call("s2e_reduce_loss_bwd", L.ptr(a), L.ptr(b), a.numel(), ctx.f32, ctx.kind, ctx.coef, 0.0, L.ptr(gout), L.ptr(da), 0, L.stream())
        if ctx.needs_input_grad[1]:     # f is even: d/db f(a - b) = d/da f(b - a)
            db = torch.empty_like(b)
            L.call("s2e_reduce_loss_bwd", L.ptr(b), L.ptr(a), a.numel(), ctx.f32, ctx.kind, ctx.coef, 0.0, L.ptr(gout), L.ptr(db), 0, L.stream())
        return da, db, None, None


def pair_mse(a, b):
    """nn.MSELoss()(a, b) with gradients to both sides."""
    return PairLossFn.apply(a, b, L.RED_L2, 1.0 / a.numel()).view(())


class AggregateFn(torch.autograd.Function):
    """Pix2PixModel._aggregate_tensor (pix2pix_model.py:271-278) over the ns style images of each sample:
    x (G * ns, ...) fp32 or bf16 (the ns images of a sample adjacent)  ->  (G, ...) fp32, mean (mode 0) or max (mode 1)."""

    @staticmethod
    def forward(ctx, x, G, ns, mode):
        x = _c(x)
        assert x.shape[0] == G * ns
        n = x.numel() // (G * ns)
        out = torch.empty((G,) + tuple(x.shape[1:]), dtype=F32, device=x.device)
        arg = torch.empty(G * n, dtype=torch.uint8, device=x.device) if mode == 1 else None
        L.call("s2e_aggregate_fwd", L.ptr(x), int(x.dtype == F32), G, ns, n, mode, L.ptr(out), L.ptr(arg), L.stream())
        ctx.dims = (G, ns, n, mode, x.shape, x.dtype)
        ctx.save_for_backward(arg)
        return out

    @staticmethod
    def backward(ctx, dout):
        G, ns, n, mode, shape, dtype = ctx.dims
        (arg,) = ctx.saved_tensors
        dout = _c(dout.float())
        dx = torch.empty(shape, dtype=dtype, device=dout.device)
        L.call("s2e_aggregate_bwd", L.ptr(dout), L.ptr(arg), int(dtype == F32), G, ns, n, mode, L.ptr(dx), L.stream())
        return dx, None, None, None


def to255_resize(images, size=(640, 400), target=None):
    """ImageProcessor.to_255resized_imagebatch (data/postprocessor.py:98-102) on the device: fp32 (N,1,h,w) in [-1,1] ->
    int32 (N,1,H,W) in [0,255] (cv2 INTER_LINEAR in float64, *255, .int(): bit-exact integers).  With an int target of the
    output's shape also returns the per-image OpenEDS score (MSECalculator.calculate_mse_for_images)."""
    x = _c(images.detach().float())
    N, C, h, w = x.shape
    H, W = size
    out = torch.empty(N, C, H, W, dtype=torch.int32, device=x.device)
    if target is None:
        L.call("s2e_to255_resize", L.ptr(x), N * C, h, w, H, W, 0, None, L.ptr(out), None, None, L.stream())
        return out
    t = _c(target.to(device=x.device, dtype=torch.int32))
    assert t.shape == out.shape
    sq = torch.empty(N * C, dtype=torch.int64, device=x.device)
    score = torch.empty(N * C, dtype=F32, device=x.device)
    L.call("s2e_to255_resize", L.ptr(x), N * C, h, w, H, W, 0, L.ptr(t), L.ptr(out), L.ptr(sq), L.ptr(score), L.stream())
    return out, score


def to255(images):
    """ImageProcessor.to_255imagebatch on an fp32 tensor (no resize, fp32 arithmetic): ((x + 1) * 255 / 2).int()."""
    x = _c(images.detach().float())
    if x.dim() == 3:
        x = x.unsqueeze(0)
    N, C, h, w = x.shape
    out = torch.empty(N, C, h, w, dtype=torch.int32, device=x.device)
    L.call("s2e_to255_resize", L.ptr(x), N * C, h, w, h, w, 1, None, L.ptr(out), None, None, L.stream())
    return out


def openeds_score(produced, target):
    """MSECalculator.calculate_mse_for_images (loss.py:113-133): per image sqrt(sum (p - t)^2) / (H * W) for two integer
    (N,1,H,W) batches in [0,255]; the sum of squares is an exact 64-bit integer."""
    p = _c(produced.to(torch.int32))
    t = _c(target.to(device=p.device, dtype=torch.int32))
    assert p.shape == t.shape and p.dim() == 4
    N, C, H, W = p.shape
    sq = torch.empty(N * C, dtype=torch.int64, device=p.device)
    score = torch.empty(N * C, dtype=F32, device=p.device)
    L.call("s2e_openeds_score", L.ptr(p), L.ptr(t), N * C, H, W, L.ptr(sq), L.ptr(score), L.stream())
    return score


# ------------------------------------------------------------------------------------------------ Gram / style loss
def _pixel_major(x_bhwc):
    """(B, h, w, C) fp32 contiguous -> (1, h, w, C*B) bf16: pixels x all (channel, sample) pairs, channel index c*B + b.
    Read as NCHW with N=1, C=B, H=h*w, W=C, this is exactly the NCHW->NHWC layout kernel."""
    B, h, w, Cc = x_bhwc.shape
    y = torch.empty(1, h, w, Cc * B, dtype=BF16, device=x_bhwc.device)
    L.call("s2e_nchw_f32_to_nhwc_bf16", L.ptr(x_bhwc), 1, B, h * w, Cc, L.ptr(y), L.stream())
    return y


def _gram_raw(xp):
    """xp (1, h, w, M) bf16 -> G[i][j] = sum_p xp[p][i] xp[p][j] (fp32, M x M): the weight-gradient GEMM of a 1x1
    convolution whose input and output gradient are both xp (pixels are the contraction axis)."""
    _, h, w, M = xp.shape
    G = torch.zeros(M * M, dtype=F32, device=xp.device)
    d = _desc(1, h, w, M, h, w, M, [(0, 0)], L.ACT_NONE)
    impl = _pick(M >= 64 and M % 8 == 0)
    flops = 2.0 * h * w * M * M
    if impl == L.IMPL_TC:
        _timed_call("tc", flops, "s2e_tapconv_wgrad", d, L.ptr(xp), L.ptr(xp), L.ptr(G), impl, L.stream(), tag="gram %dx%d M%d" % (h, w, M))
    else:
        L.call("s2e_tapconv_wgrad", d, L.ptr(xp), L.ptr(xp), L.ptr(G), impl, L.stream())
    return G.view(M, M)


class GramLossFn(torch.autograd.Function):
    """StyleLoss (loss.py:177-200) on two feature batches given as (B, h, w, C) fp32:
    mse(gram(fake), gram(real).detach()) with gram(x) = F F^T / (B*C*h*w), F = x viewed as (B*C, h*w).
    Forward: two Gram GEMMs on the tensor cores (weight-gradient kernel, K = h*w) + one reduction.  Backward:
    dF = 2 D F with D = dL/dG (symmetric), i.e. a 1x1 convolution over the same pixel-major tensor."""

    @staticmethod
    def forward(ctx, ff, fr):
        ff, fr = _c(ff.float()), _c(fr.detach().float())
        B, h, w, Cc = ff.shape
        M = B * Cc
        xf, xr = _pixel_major(ff), _pixel_major(fr)
        Gf, Gr = _gram_raw(xf), _gram_raw(xr)
        norm = float(B * Cc * h * w)
        coef = 1.0 / (norm * norm * M * M)
        out = torch.empty(1, dtype=F32, device=ff.device)
        L.call("s2e_reduce_loss", L.ptr(Gf), L.ptr(Gr), M * M, 1, L.RED_L2, coef, 0.0, L.ptr(out), 0, L.stream())
        ctx.dims, ctx.coef = (B, h, w, Cc), coef
        ctx.save_for_backward(xf, Gf, Gr)
        return out

    @staticmethod
    def backward(ctx, gout):
        xf, Gf, Gr = ctx.saved_tensors
        B, h, w, Cc = ctx.dims
        M = B * Cc
        st = L.stream()
        gout = _c(gout.float())
        D = torch.empty_like(Gf)     # dL/dG_raw = gout * coef * 2 (Gf - Gr), symmetric
        L.call("s2e_reduce_loss_bwd", L.ptr(Gf), L.ptr(Gr), M * M, 1, L.RED_L2, ctx.coef, 0.0, L.ptr(gout), L.ptr(D), 0, st)
        wp = torch.empty(M * M, dtype=BF16, device=D.device)
        L.call("s2e_pack_weight", L.ptr(D), M, M, 1, 1, 1, 0, 0, M, 0, 0, L.ptr(wp), st)
        two = torch.full((1,), 2.0, dtype=F32, device=D.device)
        dxf = torch.empty_like(xf)
        d = _desc(1, h, w, M, h, w, M, [(0, 0)], L.ACT_NONE)
        impl = _pick(M % 64 == 0)
        L.call("s2e_tapconv_fwd", d, L.ptr(xf), L.ptr(wp), None, L.ptr(two), L.ptr(dxf), impl, st)
        dff = torch.empty(B, h, w, Cc, dtype=F32, device=D.device)
        L.call("s2e_nhwc_bf16_to_nchw_f32", L.ptr(dxf), 1, B, h * w, Cc, L.ptr(dff), st)
        return dff, None


def gram_loss(ff, fr):
    return GramLossFn.apply(ff, fr).view(())


def gram_matrix(x_nchw):
    """loss.py:177-189 for an NCHW tensor (a, b, c, d) on the device: (a*b, a*b) fp32 = F F^T / (a*b*c*d) through the
    tensor-core Gram GEMM (inputs rounded to bf16)."""
    x = _c(x_nchw.detach().float())
    a, b, c, d = x.shape
    xp = torch.empty(1, c, d, a * b, dtype=BF16, device=x.device)
    L.call("s2e_nchw_f32_to_nhwc_bf16", L.ptr(x), 1, a * b, c, d, L.ptr(xp), L.stream())
    return _gram_raw(xp) / float(a * b * c * d)


# ------------------------------------------------------------------------------------------------ image head
class _ConvCtx:
    """Stand-in for an autograd ctx so that ImageHeadFn can reuse TapConvFn.backward for its convolution part."""


class ImageHeadFn(torch.autograd.Function):
    """leaky_relu(x, 0.2) -> conv_img (64 -> 1, 3x3, pad 1) -> tanh (generator.py:97-99) in ONE kernel: the activation is
    applied as the input tile is read, tanh to the fp32 accumulator (the pre-activation is never rounded to bf16), the image
    leaves as fp32 (B,1,H,W).  With `target` (the image the L1 / L2 losses compare against, pix2pix_model.py:197-208) the
    same kernel also reduces sum|fake - target| and sum (fake - target)^2 into `sums` (2,), so the image losses need no
    pass of their own over the image.  Returns (image, sums | None)."""

    @staticmethod
    def forward(ctx, x, cfg, weight, bias, target):
        x = _c(x)
        B, H, W, Cin = x.shape
        assert x.dtype == BF16 and Cin == 64 and tuple(weight.shape) == (1, 64, 3, 3) and cfg.stride == 1 and cfg.pad == 1
        taps = conv_taps(cfg)
        wp = packed_weights((weight,), cfg, False)
        img = torch.empty(B, 1, H, W, dtype=F32, device=x.device)
        sums = None
        if target is not None:
            target = _c(target.detach().float())
            assert target.shape == img.shape
            sums = torch.zeros(2, dtype=F32, device=x.device)
        d = _desc(B, H, W, 64, H, W, 1, taps, L.ACT_NONE)
        d.bias_n, d.in_act = 1, cfg.in_act
        d.img_out, d.img_target, d.img_sums = L.ptr(img), L.ptr(target), L.ptr(sums)
        L.call("s2e_tapconv_fwd", d, L.ptr(x), L.ptr(wp), L.ptr(bias.detach()) if bias is not None else None, None, None,
               L.IMPL_SIMT, L.stream())
        ctx.cfg, ctx.weight, ctx.has_bias = cfg, weight, bias is not None
        ctx.skip_wgrad = _state["skip_wgrad"]
        ctx.save_for_backward(x, img)
        if sums is not None:
            ctx.mark_non_differentiable(sums)
        return img, sums

    @staticmethod
    def backward(ctx, dimg, _dsums):
        x, img = ctx.saved_tensors
        B, H, W, _ = x.shape
        dz = torch.empty(B, H, W, 1, dtype=BF16, device=x.device)          # d tanh = 1 - y^2
        L.call("s2e_tanh_bwd", L.ptr(_c(dimg.float())), L.ptr(img), img.numel(), L.ptr(dz), L.stream())
        c = _ConvCtx()
        c.cfg, c.sn, c.n_w, c.n_b = ctx.cfg, None, 1, int(ctx.has_bias)
        c.in_shape, c.weights, c.cout, c.cp = tuple(x.shape), (ctx.weight,), 1, 1
        c.skip_wgrad, c.flops = ctx.skip_wgrad, 2.0 * B * H * W * 64 * 9
        c.saved_tensors = (x, None)
        c.needs_input_grad = (ctx.needs_input_grad[0], False, False, False, False, ctx.needs_input_grad[2]) + (
            (ctx.needs_input_grad[3],) if ctx.has_bias else ())
        res = TapConvFn.backward(c, dz)
        return res[0], None, res[5], (res[6] if ctx.has_bias else None), None


class PrecomputedLossFn(torch.autograd.Function):
    """coef * sums[idx] where sums[idx] = sum f(a - b) was already reduced by the kernel that produced `a` (ImageHeadFn);
    backward is the ordinary elementwise gradient of the loss."""

    @staticmethod
    def forward(ctx, a, b, sums, idx, kind, coef):
        ctx.kind, ctx.coef = kind, coef
        ctx.save_for_backward(a, b)
        return sums[idx:idx + 1] * coef

    @staticmethod
    def backward(ctx, gout):
        a, b = ctx.saved_tensors
        a, b = _c(a), (_c(b) if b is not None else None)
        gout = _c(gout.float())
        da = torch.empty_like(a)
        L.call("s2e_reduce_loss_bwd", L.ptr(a), L.ptr(b), a.numel(), int(a.dtype == F32), ctx.kind, ctx.coef, 0.0, L.ptr(gout),
               L.ptr(da), 0, L.stream())
        return da, None, None, None, None, None
