"""torch.optim.Adam semantics (reference pix2pix_model.py:92-110) with the update done by our fused kernel.
Step count / learning rate / bias corrections are kept in a small device array per parameter group so the whole
optimizer step is capturable in a CUDA graph (no host-side scalars baked into kernel arguments)."""
import torch

from . import _lib as L
from . import ops


def check_ema_decay(beta):
    beta = float(beta)
    if not 0.0 <= beta < 1.0:
        raise ValueError("ema_decay must be in [0, 1), got %r" % beta)
    return beta


class Adam(torch.optim.Optimizer):
    """`ema` (optional): {parameter: tensor of the same shape} -- after every step each such parameter's moving average
    advances, e <- fmaf(beta_t, e - p, p) with beta_t = min(ema_decay, (1 + t) / (10 + t)) at step count t, in the Adam
    launch itself.  `ema_buffers`: (destination, source) tensor pairs byte-copied after every step, in one more launch.
    Neither is part of the optimizer's state_dict.  The packed bf16 copies of the EMA tensors are not re-packed here
    (ops.pack_on_use): ema_written() marks them stale, and the next forward that reads them re-packs them."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, ema=None, ema_buffers=(),
                 ema_decay=0.0):
        defaults = dict(lr=lr, betas=(float(betas[0]), float(betas[1])), eps=eps, weight_decay=weight_decay)
        super().__init__(params, defaults)
        self.ema, self.ema_buffers, self.ema_decay = ema, list(ema_buffers), check_ema_decay(ema_decay)
        for p, e in (ema or {}).items():
            assert e.shape == p.shape and e.dtype == torch.float32 and e.is_contiguous()
        for d, s_ in self.ema_buffers:
            assert d.dtype == s_.dtype and d.shape == s_.shape and d.is_contiguous() and s_.is_contiguous()

    def _dev_state(self, group):
        ps = [p for p in group['params'] if p.grad is not None]
        st = group.get('_s2e_state')
        if st is None and ps:
            st = torch.tensor([0.0, group['lr'], 0.0, 0.0], dtype=torch.float32, device=ps[0].device)
            group['_s2e_state'] = st
            group['_s2e_lr'] = group['lr']
        elif st is not None and group['_s2e_lr'] != group['lr']:
            # learning-rate change (pix2pix_trainer.py:68-88): a host->device write outside any graph replay
            st[1:2].copy_(torch.tensor([group['lr']], dtype=torch.float32), non_blocking=False)
            group['_s2e_lr'] = group['lr']
        return st, ps

    def sync_hyperparams(self):
        """Push a changed learning rate to the device state (needed when steps are replayed from a CUDA graph)."""
        for group in self.param_groups:
            self._dev_state(group)

    @torch.no_grad()
    def step(self, closure=None):
        """One multi-tensor launch per 48 parameters (with the EMA update when `ema` is set, then the buffer copies), then
        one multi-tensor re-pack of the bf16 copies of the weights that just changed (ops.repack_stale) -- all capturable
        in a CUDA graph."""
        import ctypes as C
        s = L.stream()
        touched = []
        for group in self.param_groups:
            b1, b2 = group['betas']
            st, ps = self._dev_state(group)
            if not ps:
                continue
            L.call("s2e_adam_prepare", L.ptr(st), b1, b2, s)
            rows = []
            for p in ps:
                state = self.state[p]
                if len(state) == 0:
                    state['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
                assert p.is_contiguous() and p.dtype == torch.float32 and g.dtype == torch.float32
                rows.append((L.ptr(p), L.ptr(g), L.ptr(state['exp_avg']), L.ptr(state['exp_avg_sq']), p.numel(), g))
            n = len(rows)
            arr = lambda k: (C.c_void_p * n)(*[r[k] for r in rows])
            args = (n, arr(0), arr(1), arr(2), arr(3), (C.c_longlong * n)(*[r[4] for r in rows]),
                    L.ptr(st), b1, b2, group['eps'], group['weight_decay'])
            if self.ema:
                L.call("s2e_adam_multi_ema", *args, (C.c_void_p * n)(*[L.ptr(self.ema[p]) for p in ps]), self.ema_decay, s)
            else:
                L.call("s2e_adam_multi", *args, s)
            touched += ps
        if self.ema_buffers:
            n = len(self.ema_buffers)
            L.call("s2e_copy_multi", n, (C.c_void_p * n)(*[L.ptr(d) for d, _ in self.ema_buffers]),
                   (C.c_void_p * n)(*[L.ptr(s_) for _, s_ in self.ema_buffers]),
                   (C.c_longlong * n)(*[s_.numel() * s_.element_size() for _, s_ in self.ema_buffers]), s)
        self.ema_written()
        ops.mark_updated(touched)
        ops.repack_stale()

    def ema_written(self):
        """The kernel wrote the averages through raw pointers: bump their versions so that their packed copies re-pack at
        their next use.  Also called after every replay of a captured step, which runs no Python."""
        if self.ema:
            ops.mark_updated(self.ema.values())
