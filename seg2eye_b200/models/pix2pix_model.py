"""Pix2PixModel with the reference's contract (reference models/pix2pix_model.py:13-374).

Same constructor, `forward(data, mode)` modes ('generator' | 'discriminator' | 'encode_only' | 'inference'), loss
dictionary keys and tensor shapes, optimizer set-up (TTUR), loss log and checkpoint layout.  The arithmetic runs in
the seg2eye_b200 kernels; what the reference computes and then throws away is not computed here:
  * D's parameter gradients inside the generator step (zeroed by the trainer before they are ever used),
  * the gradient w.r.t. the detached fake image inside the discriminator step,
  * torch.cat copies of [seg, image] (one layout kernel builds the D input), slices of the D features for the
    feature-matching loss (evaluated on the un-split [fake ; real] tensors).
"""
import argparse
import contextlib
import copy
import os

import torch
from torch import nn

from .. import _lib as L
from .. import ops, optim, parallel, util
from . import networks


def _opt(opt, name, default=0):
    return getattr(opt, name, default)


def _diff_augment_arg(value):
    """--diff_augment: unknown ops are rejected while parsing; the value comes back in canonical order."""
    try:
        return ','.join(ops.parse_diff_augment(value)[0])
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e))


class Pix2PixModel(torch.nn.Module):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        networks.modify_commandline_options(parser, is_train)
        parser.add_argument('--ema_decay', type=float, default=0.0,
                            help='beyond the reference: keep an exponential moving average of the G and E weights with '
                                 'this decay, 0 <= decay < 1 (0: off); inference uses it, saved as <epoch>_net_G_ema.pth')
        parser.add_argument('--diff_augment', type=_diff_augment_arg, default='',
                            help='beyond the reference: differentiable augmentation of everything D sees in training '
                                 '(DiffAugment), a comma-separated subset of color,translation,cutout (always applied in '
                                 'that order; empty: off)')
        return parser

    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        self.ema_decay = optim.check_ema_decay(_opt(opt, 'ema_decay', 0.0))
        self.diffaug_ops, self.diffaug_policy = ops.parse_diff_augment(_opt(opt, 'diff_augment', ''))
        self.netG, self.netD, self.netE = self.initialize_networks(opt)
        self.netG_ema = self.netE_ema = None
        self.diffaug_state = None
        self._last_d_out = None
        if not opt.isTrain:
            return
        if self.diffaug_policy:
            # int64 [seed, draw counter] on the device: s2e_diffaug_draw reads and advances the counter there, so replays
            # of a captured step draw new parameters.  Held here, not by netD, whose state_dict keeps the reference's keys.
            seed = int(torch.randint(-2 ** 63, 2 ** 63 - 1, (), dtype=torch.int64))
            self.diffaug_state = torch.tensor([seed, 0], dtype=torch.int64, device=self.device())
        if self.ema_decay > 0:
            self._initialize_ema(opt)
        if not _opt(opt, 'no_vgg_loss', True):
            raise ValueError('VGG loss does not exist in the reference either (networks.VGGLoss is undefined)')
        self.criterionGAN = networks.GANLoss(opt.gan_mode, opt=opt)
        self.criterionFeat = self.criterionL1 = networks.l1_loss
        self.criterionL2 = networks.mse_loss
        self.criterionOpenEDS = networks.MSECalculator.calculate_mse_for_tensors
        self.criterion_style_feat = self.criterion_style_w = ops.pair_mse
        if _opt(opt, 'lambda_gram') > 0:
            self.criterion_gram = networks.StyleLoss()
        self.reset_loss_log()

    # ------------------------------------------------------------------ bookkeeping
    def get_loss_log(self):
        return {k: torch.stack(v).mean() for k, v in self.loss_log.items() if v}

    def add_to_loss_log(self, key, value):
        self.loss_log.setdefault(key, []).append(value)

    def reset_loss_log(self):
        self.loss_log = {}

    def use_gpu(self):
        return len(self.opt.gpu_ids) > 0

    def device(self):
        return next(self.netG.parameters()).device

    def save(self, epoch):
        self.sync_ema()
        for net, tag in ((self.netG, 'G'), (self.netD, 'D'), (self.netE, 'E'), (self.netG_ema, 'G_ema'), (self.netE_ema, 'E_ema')):
            if net is not None:
                util.save_network(net, tag, epoch, self.opt)

    def initialize_networks(self, opt):
        netG = networks.define_G(opt)
        netD = networks.define_D(opt) if opt.isTrain else None
        # --netG spade: the original style-less SPADE generator (BASELINE config 5) has no style encoder
        netE = networks.define_E(opt) if _opt(opt, 'netG', 'spadestyle') != 'spade' else None
        if not opt.isTrain or opt.continue_train:
            # a model trained with --ema_decay is tested with the averaged generator
            util.load_network(netG, 'G_ema' if not opt.isTrain and self.ema_decay > 0 else 'G', opt.which_epoch, opt)
            if opt.isTrain:   # like the reference, test time keeps a freshly initialised style encoder
                util.load_network(netD, 'D', opt.which_epoch, opt)
                if netE is not None:
                    util.load_network(netE, 'E', opt.which_epoch, opt)
        return netG, netD, netE

    # ------------------------------------------------------------------ exponential moving average (--ema_decay)
    def _initialize_ema(self, opt):
        """netG_ema / netE_ema: frozen copies of netG / netE (or, on --continue_train, the saved averages when they exist)
        that optimizer_G's Adam launch advances.  Their bf16 packed copies are refreshed by the first forward that reads
        them after a G step (optim.Adam.ema_written), not by the training step (ops.pack_on_use)."""
        def frozen_copy(net):
            ema = copy.deepcopy(net, {id(opt): opt}).requires_grad_(False)
            ops.pack_on_use(list(ema.parameters()))
            return ema
        self.netG_ema = frozen_copy(self.netG)
        self.netE_ema = frozen_copy(self.netE) if self.netE is not None else None
        if opt.continue_train:
            for _, ema, tag in self._ema_pairs():
                if os.path.exists(os.path.join(opt.checkpoints_dir, opt.name, '%s_net_%s_ema.pth' % (opt.which_epoch, tag))):
                    util.load_network(ema, tag + '_ema', opt.which_epoch, opt)
        self._ema_stale = False
        for live, _, _ in self._ema_pairs():     # weights loaded into G / E from now on restart their averages
            live.register_load_state_dict_post_hook(self._live_weights_replaced)

    def _live_weights_replaced(self, module, incompatible_keys):
        self._ema_stale = True

    def _ema_pairs(self):
        if self.netG_ema is None:
            return []
        return [(live, ema, tag) for live, ema, tag in ((self.netG, self.netG_ema, 'G'), (self.netE, self.netE_ema, 'E'))
                if ema is not None]

    @torch.no_grad()
    def reset_ema(self):
        """netG_ema / netE_ema <- netG / netE (parameters and buffers), in place: captured CUDA graphs keep their pointers."""
        for live, ema, _ in self._ema_pairs():
            for a, b in zip(list(ema.parameters()) + list(ema.buffers()), list(live.parameters()) + list(live.buffers())):
                a.copy_(b)
        self._ema_stale = False

    def sync_ema(self):
        """Restart the averages from the live nets if weights were loaded into G / E since (load_state_dict)."""
        if self.netG_ema is not None and self._ema_stale:
            self.reset_ema()

    def ema_targets(self):
        """optim.Adam's EMA arguments for the G+E optimizer: {parameter: average} and (EMA buffer, live buffer) pairs."""
        pairs = self._ema_pairs()
        ema = {p: e for live, em, _ in pairs for p, e in zip(live.parameters(), em.parameters())}
        bufs = [(e, b) for live, em, _ in pairs for b, e in zip(live.buffers(), em.buffers())]
        return dict(ema=ema, ema_buffers=bufs, ema_decay=self.ema_decay) if pairs else {}

    @contextlib.contextmanager
    def _inference_nets(self):
        """The inference modes run netG_ema / netE_ema, when they exist, in place of netG / netE."""
        if self.netG_ema is None:
            yield
            return
        self.sync_ema()
        live = self.netG, self.netE
        self.netG, self.netE = self.netG_ema, self.netE_ema
        try:
            yield
        finally:
            self.netG, self.netE = live

    def create_optimizers(self, opt):
        """Adam over G+E and over D; TTUR (default) = betas (0, 0.9), lr/2 for G, lr*2 for D."""
        if opt.no_TTUR:
            betas, g_lr, d_lr = (opt.beta1, opt.beta2), opt.lr, opt.lr
        else:
            betas, g_lr, d_lr = (0, 0.9), opt.lr / 2, opt.lr * 2
        wd = _opt(opt, 'weight_decay', 0.0)
        g_params = list(self.netG.parameters()) + (list(self.netE.parameters()) if self.netE is not None else [])
        d_params = list(self.netD.parameters()) if opt.isTrain else []
        return (optim.Adam(g_params, lr=g_lr, betas=betas, weight_decay=wd, **self.ema_targets()),
                optim.Adam(d_params, lr=d_lr, betas=betas, weight_decay=wd))

    # ------------------------------------------------------------------ entry point
    def forward(self, data, mode):
        seg, style, target = self.preprocess_input(data)
        if mode == 'generator':
            return self.compute_generator_loss(seg, style, target)
        if mode == 'discriminator':
            return self.compute_discriminator_loss(seg, style, target)
        if mode == 'encode_only':
            with self._inference_nets():
                return self.encode_w(style)[0]
        if mode == 'inference':
            with torch.no_grad(), self._inference_nets():
                if 'latent_style' in data:
                    fake = self.generate_fake_from_stylecode(seg, data['latent_style'].to(seg.device))
                else:
                    fake = self.generate_fake(seg, style)[0]
                self.reset_loss_log()
            return fake
        raise ValueError("|mode| is invalid")

    def preprocess_input(self, data):
        """label -> int64 on the device -> one-hot (B, label_nc, H, W); `data` is updated in place like the reference's."""
        dev = self.device()
        data['label'] = data['label'].long().to(dev, non_blocking=True)
        if 'style_image' in data:      # (absent for the style-less generator, --netG spade)
            data['style_image'] = data['style_image'].to(dev, non_blocking=True)
        lab = data['label']
        if lab.dim() == 3:   # (B,H,W) as the data loader collates it; the reference only handles B == 1 here
            lab = lab.unsqueeze(0) if lab.shape[0] == 1 else lab.unsqueeze(1)
        seg = ops.one_hot(lab, self.opt.label_nc)
        target = None
        if 'target' in data:
            target = data['target'] = data['target'].to(dev, non_blocking=True)
        return seg, data.get('style_image'), target

    # ------------------------------------------------------------------ losses
    def compute_generator_loss(self, input_semantics, style_image, target_image):
        opt = self.opt
        if (opt.lambda_l1 or opt.lambda_l2) and target_image is not None:
            # the image head of the generator reduces the L1 / L2 sums against this target in its own kernel
            target_image = target_image.float().contiguous()
            self.netG.loss_target = target_image
        fake, w_real, feats_real = self.generate_fake(input_semantics, style_image)
        with ops.skip_weight_grads():
            if opt.no_ganFeat_loss:
                pred_fake, pred_real = self.discriminate(input_semantics, fake, target_image)
            else:
                with ops.fm_pair_sums():    # D's InstanceNorm kernels also reduce the feature-matching L1 of their [fake ; real] output
                    pred_fake, pred_real = self.discriminate(input_semantics, fake, target_image)
        d_full, self._last_d_out = self._last_d_out, None
        losses = {'GAN': self.criterionGAN(pred_fake, True, for_discriminator=False)}
        for key, lam, crit in (('L2', opt.lambda_l2, self.criterionL2), ('L1', opt.lambda_l1, self.criterionL1)):
            if lam:
                raw = crit(fake, target_image)
                losses[key + '/weighted'] = raw * lam
                self.add_to_loss_log(key + '/raw', raw.detach())
        if _opt(opt, 'lambda_openeds'):
            # (B,) values without a gradient: ImageProcessor.to_255imagebatch ends in .int() (postprocessor.py:72), so in the
            # reference too this term only shifts the reported loss
            raw = self.criterionOpenEDS(fake.detach(), target_image)
            losses['openeds/weighted'] = raw * opt.lambda_openeds
            self.add_to_loss_log('openeds/raw', raw)
        if _opt(opt, 'lambda_style_feat') or _opt(opt, 'lambda_style_w') or _opt(opt, 'lambda_gram'):
            w_fake, feats_fake = self.encode_w(fake.unsqueeze(1))
            extra = []
            if opt.lambda_style_w > 0:
                extra.append(('style_w', opt.lambda_style_w, self.criterion_style_w(w_fake, w_real)))
            if opt.lambda_style_feat > 0:
                extra.append(('style_feat', opt.lambda_style_feat, self._compute_style_feature_loss(feats_fake, feats_real)))
            if opt.lambda_gram > 0:
                extra.append(('gram', opt.lambda_gram, self._compute_gram_loss(feats_fake, feats_real)))
            for key, lam, raw in extra:
                losses[key + '/weighted'] = raw * lam
                self.add_to_loss_log(key + '/raw', raw.detach())
        if not opt.no_ganFeat_loss:
            n_scales = len(pred_fake)
            fm = torch.zeros(1, device=fake.device)
            for i in range(n_scales):
                for j in range(len(pred_fake[i]) - 1):      # the last entry is the prediction itself
                    if d_full is not None:                   # L1(fake half, real half.detach()) on the un-split tensor
                        t = networks.loss._flat(d_full[i][j])
                        pre = getattr(d_full[i][j], '_s2e_fm_sum', None)   # reduced by the InstanceNorm kernel that produced it
                        if pre is not None and t is d_full[i][j] and pre[1] == t._version:
                            term = ops.HalvesPresummedFn.apply(t, pre[0], L.RED_L1, 2.0 / t.numel()).view(())
                        else:
                            term = ops.HalvesLossFn.apply(t, L.RED_L1, 2.0 / t.numel()).view(())
                    else:
                        term = self.criterionFeat(pred_fake[i][j], pred_real[i][j].detach())
                    fm = fm + term * opt.lambda_feat / n_scales
            losses['GAN_Feat'] = fm
        return losses, fake

    def compute_discriminator_loss(self, input_semantics, real_image, target_image):
        with torch.no_grad():   # E and G run again, in training mode: BN running stats and u/v advance once more
            fake = self.generate_fake(input_semantics, real_image)[0].detach()
        pred_fake, pred_real = self.discriminate(input_semantics, fake, target_image)
        self._last_d_out = None   # never keep an autograd graph alive across steps (CUDA-graph capture relies on it)
        return {'D/Fake': self.criterionGAN(pred_fake, False, for_discriminator=True),
                'D/real': self.criterionGAN(pred_real, True, for_discriminator=True)}

    def _compute_style_feature_loss(self, features_fake, features_real):
        """pix2pix_model.py:162-172: sum over the encoder levels of MSE(aggregated fake features, aggregated real
        features) -- nothing is detached in the reference, so both sides receive gradients."""
        return torch.stack([ops.pair_mse(f, r) for f, r in zip(features_fake, features_real)]).sum()

    def _compute_gram_loss(self, features_fake, features_real):
        """pix2pix_model.py:174-184 + loss.py:177-200: per level MSE of the Gram matrices of the (B*C, h*w) feature
        matrices, the real side detached (loss.py:198)."""
        return torch.stack([self.criterion_gram(f, r, nhwc=True) for f, r in zip(features_fake, features_real)]).sum()

    # ------------------------------------------------------------------ style encoder
    def _aggregate_mode(self):
        how = self.opt.style_aggr_method
        if how not in ('mean', 'max'):
            raise ValueError(f"Aggregation method not found: {how}")
        return 0 if how == 'mean' else 1

    def _aggregate_tensor(self, tensor, dim=1):
        """pix2pix_model.py:271-278 for a (G, ns, ...) tensor along dim 1 or a (ns, ...) tensor along dim 0."""
        mode = self._aggregate_mode()
        if dim == 0:
            return ops.AggregateFn.apply(tensor, 1, tensor.shape[0], mode)[0]
        assert dim == 1
        G, ns = tensor.shape[:2]
        return ops.AggregateFn.apply(tensor.reshape(G * ns, *tensor.shape[2:]), G, ns, mode)

    def _compute_multiple_netE(self, real_image):
        """(B, ns, 1, H, W) -> mu (B, ns, w_dim) and the encoder's feature maps, each (B*ns, C, h, w).  The reference calls
        netE once per sample, advancing its spectral-norm vectors once per call; ConvEncoder.forward_samples reproduces
        exactly that in one batched pass."""
        n_b, ns = real_image.shape[:2]
        mu, _, feats = self.netE.forward_samples(real_image)
        assert mu.shape == (n_b, ns, self.opt.w_dim)
        return mu, feats

    def _compute_aggregated_w(self, real_image):
        """-> w (B, w_dim) and, when a style-feature / Gram loss needs them, one aggregated feature map per encoder level,
        (B, h, w, C) fp32 (the reference keeps a per-sample list of (C, h, w) maps and stacks them per level later)."""
        mu, feats = self._compute_multiple_netE(real_image)
        w = self._aggregate_tensor(mu)
        agg = []
        if self.opt.isTrain and (_opt(self.opt, 'lambda_style_feat') or _opt(self.opt, 'lambda_gram')):
            n_b, ns = real_image.shape[:2]
            agg = [ops.AggregateFn.apply(ops.as_nhwc(f), n_b, ns, self._aggregate_mode()) for f in feats]
        return w, agg

    def encode_w(self, real_image):
        if real_image.dim() != 5:
            raise ValueError("real_image should have 5 dimensions")
        return self._compute_aggregated_w(real_image)

    def generate_fake_from_stylecode(self, input_semantics, latent_style):
        return self.netG(input_semantics, latent_style)

    def generate_fake(self, input_semantics, style_image):
        if self.netE is None:       # plain SPADE generator: no style code
            return self.netG(input_semantics), None, []
        w, feats = self.encode_w(style_image)
        return self.generate_fake_from_stylecode(input_semantics, w), w, feats

    # ------------------------------------------------------------------ discriminator call
    def discriminate(self, input_semantics, fake_image, real_image):
        """cat([seg,fake],1) / cat([seg,real],1) / cat(.,0) of the reference as ONE layout kernel; channels are
        zero-padded to 16 so that D's first 4x4-s2 convolution is tensor-core shaped after space-to-depth.
        With --diff_augment, in training, the layout kernel's augmented twin builds it: one parameter record per sample
        pair (fake b and real b alike, so the feature-matching loss still compares aligned images), drawn for the
        sample's global index rank * B + b."""
        # (5 -> 16 channels for the 4-class OpenEDS maps; in general the next multiple of 16)
        cpad = -(-(input_semantics.shape[1] + 1) // 16) * 16
        if self.diffaug_policy and self.training:
            B, _, H, W = input_semantics.shape
            params = ops.diffaug_draw(self.diffaug_state, B, parallel.rank() * B, H, W)
            both = ops.MakeDInputAugFn.apply(input_semantics, fake_image, real_image, cpad, params, self.diffaug_policy)
        else:
            both = ops.MakeDInputFn.apply(input_semantics, fake_image, real_image, cpad)
        out = self.netD.forward_nhwc(both)
        self._last_d_out = out
        return self.divide_pred(out)

    def divide_pred(self, pred):
        def halves(t):
            n = t.size(0) // 2
            a, b = t[:n], t[n:]
            sums = getattr(t, '_s2e_gan_sums', None)    # logits whose gather kernel already reduced both halves (ops.head_conv)
            if sums is not None and t.size(0) == 2 * n:
                a._s2e_gan_half, b._s2e_gan_half = (sums, 0, a._version), (sums, 1, b._version)
            return a, b
        if isinstance(pred, list):
            split = [[halves(t) for t in scale] for scale in pred]
            return [[p[0] for p in s] for s in split], [[p[1] for p in s] for s in split]
        return halves(pred)
