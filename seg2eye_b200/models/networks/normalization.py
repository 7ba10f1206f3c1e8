"""SPADE / ApplyStyle / SPADE_STYLE_Block mirrors (reference models/networks/normalization.py)."""
import re

import torch
import torch.nn as nn

from ... import _lib as L
from ... import ops
from .layers import BatchNorm2dStats, Conv2d, InstanceNorm2d


def get_nonspade_norm_layer(opt, norm_type='instance'):
    """normalization.py:15-47: wrap a conv in spectral norm, drop its bias, append the sub-norm.
    Returns nn.Sequential(conv, norm) (or the bare conv for 'spectralnone')."""
    def add_norm_layer(layer):
        if not norm_type.startswith('spectral'):
            # the reference leaves subnorm_type undefined here and crashes (normalization.py:25-29)
            raise ValueError('normalization layer %s is not recognized' % norm_type)
        subnorm_type = norm_type[len('spectral'):]
        has_bias = subnorm_type == 'none' or len(subnorm_type) == 0
        cfg = layer.cfg
        layer = Conv2d(layer.in_channels, layer.out_channels, cfg.kh, stride=cfg.stride, padding=cfg.pad,
                       bias=has_bias and layer.bias is not None, spectral=True)
        if has_bias:
            return layer
        if subnorm_type == 'instance':
            norm_layer = InstanceNorm2d(layer.out_channels)
        elif subnorm_type == 'batch':
            raise ValueError('normalization layer batch is not supported by the B200 path (reference default is instance)')
        else:
            raise ValueError('normalization layer %s is not recognized' % subnorm_type)
        return nn.Sequential(layer, norm_layer)
    return add_norm_layer


_col_cache = {"key": None, "cols": {}}


def seg_im2col_cached(segmap, h, w):
    """im2col of `segmap` at (h, w), memoised for as long as the same segmap tensor object (and version) is in use."""
    key = (id(segmap), segmap._version, segmap.data_ptr(), tuple(segmap.shape))
    if _col_cache["key"] != key or (_col_cache.get("ref") is None or _col_cache["ref"]() is not segmap):
        import weakref
        _col_cache["key"], _col_cache["cols"] = key, {}
        _col_cache["ref"] = weakref.ref(segmap)
    cols = _col_cache["cols"]
    if (h, w) not in cols:
        cols[(h, w)] = ops.seg_im2col(segmap, h, w)
    return cols[(h, w)]


def seg_nearest_cached(segmap, h, w, cpad):
    """Nearest-resized (and channel-padded) segmap at (h, w), shared by the SPADE blocks of one generator forward."""
    key = (id(segmap), segmap._version, segmap.data_ptr(), tuple(segmap.shape))
    if _col_cache["key"] != key or (_col_cache.get("ref") is None or _col_cache["ref"]() is not segmap):
        import weakref
        _col_cache["key"], _col_cache["cols"] = key, {}
        _col_cache["ref"] = weakref.ref(segmap)
    cols = _col_cache["cols"]
    if ("nearest", h, w, cpad) not in cols:
        cols[("nearest", h, w, cpad)] = ops.seg_nearest(segmap, h, w, cpad)
    return cols[("nearest", h, w, cpad)]


def clear_seg_cache():
    """Called at both ends of a generator forward: the resized / im2col'd segmaps and the shared statistics sums (ops) live for one
    forward only, so nothing cached can outlive the tensors (or the CUDA-graph capture) it was computed from."""
    _col_cache["key"], _col_cache["cols"] = None, {}
    ops.clear_stats_memo()


class FC(nn.Module):
    """normalization.py:108-141 (StyleGAN dense layer + LeakyReLU(0.2))."""

    def __init__(self, in_channels, out_channels, gain=2 ** 0.5, use_wscale=False, lrmul=1.0, bias=True):
        super().__init__()
        he_std = gain * in_channels ** (-0.5)
        if use_wscale:
            init_std = 1.0 / lrmul
            self.w_lrmul = he_std * lrmul
        else:
            init_std = he_std / lrmul
            self.w_lrmul = lrmul
        self.weight = nn.Parameter(torch.randn(out_channels, in_channels) * init_std)
        if bias:
            self.bias = nn.Parameter(torch.zeros(out_channels))
            self.b_lrmul = lrmul
        else:
            self.bias = None

    def forward(self, x):
        w = self.weight if self.w_lrmul == 1.0 else self.weight * self.w_lrmul
        b = self.bias
        if b is not None and self.b_lrmul != 1.0:
            b = b * self.b_lrmul
        return ops.LinearFn.apply(x.float(), w, b, L.ACT_LRELU, 0)


class ApplyStyle(nn.Module):
    """normalization.py:144-169: x * (style[:,0] + 1) + style[:,1] with style = FC(w)."""

    def __init__(self, latent_size, channels, use_wscale):
        super().__init__()
        self.linear = FC(latent_size, channels * 2, gain=1.0, use_wscale=use_wscale)

    def forward(self, x, latent_style):
        # standalone use (the fused block below never materialises this): gamma = beta = 0, no norm => 2*(0.5*x*(1+s0)+...)
        style = self.linear(latent_style)
        xn = ops.as_nhwc(x)
        B, H, W, C = xn.shape
        gb = torch.zeros(B, H, W, 2 * C, dtype=torch.bfloat16, device=xn.device)
        # identity norm (mean 0, rstd 0 kills the SPADE term), doubled style so that 0.5*(...) gives x*(1+s0)+s1
        st2 = torch.cat([2 * style[:, :C] + 1, 2 * style[:, C:]], dim=1)
        cfg = ops.NormCfg(False, L.ACT_NONE, False, 0.0, 1e-5)
        rm = torch.zeros(C, device=xn.device)
        rv = torch.full((C,), float('inf'), device=xn.device)
        return ops.as_nchw_view(ops.SpadeStyleFn.apply(xn, gb, st2, cfg, rm, rv, None))


class SPADE(nn.Module):
    """normalization.py:63-105.  gamma and beta are produced by ONE implicit GEMM with N = 2C (their weights
    are packed side by side), then consumed by the fused normalisation/modulation kernel."""

    def __init__(self, config_text, norm_nc, label_nc):
        super().__init__()
        assert config_text.startswith('spade')
        parsed = re.search(r'spade(\D+)(\d)x\d', config_text)
        param_free_norm_type = str(parsed.group(1))
        ks = int(parsed.group(2))
        if param_free_norm_type == 'instance':
            self.param_free_norm = InstanceNorm2d(norm_nc)
            self.per_sample = True
        elif param_free_norm_type in ('batch', 'syncbatch'):
            # syncbatch (the reference SPADE's default, rejected by Seg2Eye): torch.nn.SyncBatchNorm(affine=False) --
            # training-mode statistics of the global batch across the ranks of the default process group; the same
            # buffers (and state_dict) as batch, and the same computation with one rank or in eval mode
            self.param_free_norm = BatchNorm2dStats(norm_nc)
            self.per_sample = False
        else:
            raise ValueError('%s is not a recognized param-free norm type in SPADE' % param_free_norm_type)
        nhidden = 128
        pw = ks // 2
        self.mlp_shared = nn.Sequential(Conv2d(label_nc, nhidden, ks, padding=pw, act=L.ACT_RELU), nn.ReLU())
        self.mlp_gamma = Conv2d(nhidden, norm_nc, ks, padding=pw)
        self.mlp_beta = Conv2d(nhidden, norm_nc, ks, padding=pw)
        self.norm_nc = norm_nc
        self.sync = param_free_norm_type == 'syncbatch'

    def _actv(self, segmap, h, w):
        """ReLU(mlp_shared(nearest(segmap))) and whether its ReLU backward is left to the gamma|beta data gradient."""
        conv = self.mlp_shared[0]
        if 9 * conv.in_channels <= 62 and conv.cfg.kh == 3:
            # thin segmap: its 64-channel im2col (shared by every SPADE of this resolution within one generator
            # forward) turns mlp_shared into a K=64 GEMM on the tensor-core path, forward and weight gradient
            col = seg_im2col_cached(segmap, h, w)
            return ops.SegConvFn.apply(col, conv.weight, conv.bias, L.ACT_RELU, True), True
        # wide label maps (e.g. 35 classes): channels zero-padded to a multiple of 64 so that mlp_shared is an ordinary
        # tap convolution on the tensor cores, forward and weight gradient (K = 9 * 64)
        cpad = -(-conv.in_channels // 64) * 64 if conv.in_channels >= 16 else 0
        return conv.forward_nhwc(seg_nearest_cached(segmap, h, w, cpad)), False

    def gamma_beta(self, segmap, h, w):
        actv, fused_relu = self._actv(segmap, h, w)
        # (the ReLU backward of actv is fused into the gamma|beta data-gradient epilogue: relu_in)
        cfg = self.mlp_gamma.cfg._replace(relu_in=True) if fused_relu else self.mlp_gamma.cfg
        return ops.tap_conv(actv, cfg, (self.mlp_gamma.weight, self.mlp_beta.weight), (self.mlp_gamma.bias, self.mlp_beta.bias))

    def modulate(self, x, segmap, style, act, up=False, sink=None):
        """x NHWC bf16; style (B,2C) fp32 (s0|s1) ->  act(0.5*[norm(x)(1+gamma)+beta + x(1+s0)+s1]);
        style None -> plain SPADE: act(norm(x)(1+gamma)+beta)  (normalization.py:91-105).
        up: x is the half-resolution tensor whose nearest-2x up-sampling is the real input (never materialised)."""
        B, H, W, C = x.shape
        if up:
            H, W = 2 * H, 2 * W
        pfn = self.param_free_norm
        cfg = ops.NormCfg(self.per_sample, act, self.training, 0.1, 1e-5, self.sync)
        bufs = (None, None, None) if self.per_sample else (pfn.running_mean, pfn.running_var, pfn.num_batches_tracked)
        if not torch.is_grad_enabled() and ops.spade_conv_fused_ok(x, up, self.mlp_gamma.in_channels):
            # no autograd graph wanted (D step's generator pass, inference): gamma|beta are consumed in the epilogue of
            # their own convolution and never written
            actv, _ = self._actv(segmap, H, W)
            return ops.spade_conv_fused(actv, self.mlp_gamma.cfg, (self.mlp_gamma.weight, self.mlp_beta.weight),
                                        (self.mlp_gamma.bias, self.mlp_beta.bias), x, style, cfg, *bufs, up)
        if (self.training and not self.per_sample and ops._state["fuse_spade_training"]
                and ops.spade_conv_fused_ok(x, up, self.mlp_gamma.in_channels)):
            # (InstanceNorm statistics -- `spadeinstance` -- keep the two-kernel path in training mode: the fused training
            #  kernel has only been validated on hardware with BatchNorm statistics so far)
            # training: same fusion, the kernel additionally keeps gamma and the activation mask for backward
            actv, fused_relu = self._actv(segmap, H, W)
            ccfg = self.mlp_gamma.cfg._replace(relu_in=True) if fused_relu else self.mlp_gamma.cfg
            return ops.SpadeConvFn.apply(actv, x, style, self.mlp_gamma.weight, self.mlp_beta.weight, self.mlp_gamma.bias,
                                         self.mlp_beta.bias, ccfg, cfg, *bufs, up, sink)
        gb = self.gamma_beta(segmap, H, W)
        return ops.SpadeStyleFn.apply(x, gb, style, cfg, *bufs, up, sink)

    def forward(self, x, segmap):
        return ops.as_nchw_view(self.modulate(ops.as_nhwc(x), segmap, None, L.ACT_NONE))


class SPADE_Block(nn.Module):
    """The style-less counterpart of SPADE_STYLE_Block for the plain SPADE generator (BASELINE config 5): the block of
    normalization.py:172-192 with the ApplyStyle half and the division by two removed, i.e. SPADE alone.  Same
    `.spade.*` parameter names, no `.adain.*`."""

    def __init__(self, fin, opt):
        super().__init__()
        self.spade = SPADE(opt.norm_G.replace('spectral', ''), fin, opt.semantic_nc)

    def forward_nhwc(self, x, segmap, latent_style=None, act=L.ACT_NONE, up=False, sink=None):
        return self.spade.modulate(x, segmap, None, act, up, sink)

    def forward(self, x, segmap, latent_style=None):
        return ops.as_nchw_view(self.forward_nhwc(ops.as_nhwc(x), segmap))


class SPADE_STYLE_Block(nn.Module):
    """normalization.py:172-192: (SPADE(x, seg) + ApplyStyle(x, w)) / 2 in one fused pass."""

    def __init__(self, fin, opt):
        super().__init__()
        spade_config_str = opt.norm_G.replace('spectral', '')
        self.spade = SPADE(spade_config_str, fin, opt.semantic_nc)
        self.adain = ApplyStyle(opt.w_dim, channels=fin, use_wscale=False)

    def forward_nhwc(self, x, segmap, latent_style, act=L.ACT_NONE, up=False, sink=None):
        """up: x is given at half resolution, its nearest-2x up-sampling is the input (read through an index map).
        sink: ops.GradSink shared with the other SPADE_STYLE_Block that reads the same x (one gradient buffer)."""
        style = self.adain.linear(latent_style)
        return self.spade.modulate(x, segmap, style, act, up, sink)

    def forward(self, x, segmap, latent_style):
        return ops.as_nchw_view(self.forward_nhwc(ops.as_nhwc(x), segmap, latent_style))
