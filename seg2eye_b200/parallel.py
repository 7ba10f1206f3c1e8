"""Data parallelism: one process per GPU, full replicas, batch sharded, per-rank BatchNorm statistics (what the
reference's nn.DataParallel did, SURVEY.md 8(e)); the only collective is the gradient average -- unless the SPADE layers
share their statistics across ranks (`--norm_G spectralspadesyncbatch3x3`, ops.synced), which adds an all-gather per
distinct SPADE input in forward and an all-reduce per SPADE layer in backward on the default group.

GradReducer averages gradients with bucketed all-reduces that OVERLAP the backward pass: every parameter carries a
post-accumulate-grad hook that copies its gradient into its bucket's flat fp32 buffer; when the last gradient of a
bucket has arrived the bucket's all-reduce is launched asynchronously (NCCL runs it on its own stream after the work
already queued on ours, so it proceeds while the remaining backward kernels run).  `allreduce()` after backward waits
for the buckets and scatters the averaged values back into `.grad`.  Buckets are built from the parameters that
actually received a gradient in the first step (fc_var never does; D's parameters get none inside the G step), in
reverse registration order ~ the order in which backward produces them.  NCCL over NVLink on the box, gloo in the CPU
tests."""
import torch
import torch.distributed as dist


def world_size():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


class _Bucket:
    __slots__ = ("params", "offsets", "flat", "pending", "handle")

    def __init__(self, params):
        self.params = params
        self.offsets, n = [], 0
        for p in params:
            self.offsets.append(n)
            n += p.numel()
        self.flat = torch.zeros(n, dtype=torch.float32, device=params[0].device)
        self.pending = len(params)
        self.handle = None


class GradReducer:
    def __init__(self, params, bucket_bytes=None, overlap=None):
        self.params = [p for p in params if p.requires_grad]
        if bucket_bytes is None:
            # S2E_BUCKET_MB: size of the flat gradient buffers.  The all-reduce runs between the two CUDA graphs of a step (nothing
            # to overlap with), so buckets only need to be large enough for NCCL's peak bus bandwidth: 8 x B200, 396 MB of G + E
            # gradients: 102.0 ms/step with 32 MB buckets, 100.4 with 128 MB, 100.3 with 512 MB (profiles/r02f_bench_n8_c2*.json)
            import os
            bucket_bytes = int(os.environ.get("S2E_BUCKET_MB", "128")) << 20
        self.bucket_bytes = bucket_bytes
        # overlap = launch each bucket's all-reduce from inside backward (post-accumulate hooks).  Off by default since round 2:
        # the CUDA-graph steps (the fast path) cannot use it, and under torch 2.11 the hooks were seen to run for parameters
        # whose gradient had not been set, which desynchronises the ranks' collective order.  S2E_OVERLAP_ALLREDUCE=1 enables it.
        if overlap is None:
            import os
            overlap = os.environ.get("S2E_OVERLAP_ALLREDUCE", "0") == "1"
        self.overlap = overlap
        self.buckets = None
        self._slot = {}
        self._hooks = []
        self.launched_during_backward = 0   # diagnostics: buckets whose all-reduce started from a hook
        self.flat_bound = False
        # Autograd runs a parameter's post-accumulate hooks even when the gradient that reached it is undefined (e.g. D's
        # parameters inside the generator step, whose weight gradients are skipped): a reducer only listens while its own
        # step is running (`armed`), and never to a parameter without a gradient
        self.armed = True

    # ---- bucket construction (first step: we now know which parameters receive gradients)
    def _build(self):
        live = [p for p in reversed(self.params) if p.grad is not None]
        self.buckets, cur, size = [], [], 0
        for p in live:
            n = p.numel() * 4
            if cur and size + n > self.bucket_bytes:
                self.buckets.append(_Bucket(cur))
                cur, size = [], 0
            cur.append(p)
            size += n
        if cur:
            self.buckets.append(_Bucket(cur))
        for bi, b in enumerate(self.buckets):
            for pi, p in enumerate(b.params):
                self._slot[p] = (bi, pi)
        if self.overlap:
            for p in live:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))

    def _on_grad(self, p):
        if not self.armed or p.grad is None:
            return
        bi, pi = self._slot[p]
        b = self.buckets[bi]
        off = b.offsets[pi]
        b.flat[off:off + p.numel()].copy_(p.grad.detach().reshape(-1))
        b.pending -= 1
        if b.pending == 0:
            b.handle = dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, async_op=True)
            self.launched_during_backward += 1

    # ---- CUDA-graph mode: gradients live INSIDE the flat buckets ------------------------------------------------
    def remove_hooks(self):
        """Stop launching all-reduces from inside backward (allreduce() then gathers the gradients itself)."""
        for h in self._hooks:
            h.remove()
        self._hooks = []
        for b in self.buckets or []:
            b.pending, b.handle = len(b.params), None

    def bind_flat_grads(self):
        """After one eager step (which tells us which parameters receive gradients): make every such parameter's .grad a
        view into its bucket's flat buffer and drop the hooks.  Backward then accumulates straight into the buckets
        (no copy-in), `allreduce_flat()` reduces them in place (no copy-out) and Adam reads the views.  The caller zeroes
        the buckets (`zero_flat()`) at the start of every step instead of setting .grad to None."""
        if self.buckets is None:
            self._build()
        self.remove_hooks()
        for b in self.buckets:
            for p, off in zip(b.params, b.offsets):
                p.grad = b.flat[off:off + p.numel()].view_as(p)
        self.flat_bound = True

    def unbind_flat_grads(self):
        """Back to eager mode: gradients become ordinary per-parameter tensors again, the overlap hooks return."""
        self.flat_bound = False
        for b in self.buckets or []:
            for p in b.params:
                p.grad = None
            b.pending, b.handle = len(b.params), None
        if self.overlap and self.buckets:
            for b in self.buckets:
                for p in b.params:
                    self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))

    def zero_flat(self):
        for b in self.buckets:
            b.flat.zero_()

    def allreduce_flat(self):
        """SUM all-reduce of the buckets in place; the 1/world_size factor is folded into the loss by the caller."""
        if world_size() == 1:
            return
        hs = [dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, async_op=True) for b in self.buckets]
        for h in hs:
            h.wait()

    # ---- called once after backward
    def allreduce(self):
        ws = world_size()
        if ws == 1:
            return
        if self.flat_bound:
            raise RuntimeError("GradReducer: gradients are bound to the flat buckets (CUDA-graph mode); use allreduce_flat()")
        first = self.buckets is None
        if first:
            self._build()
        for b in self.buckets:
            if b.handle is None:
                # first step (hooks were not installed yet) or a gradient that did not arrive: gather what exists
                for p, off in zip(b.params, b.offsets):
                    if p.grad is not None:
                        b.flat[off:off + p.numel()].copy_(p.grad.detach().reshape(-1))
                    else:
                        b.flat[off:off + p.numel()].zero_()
                b.handle = dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, async_op=True)
        inv = 1.0 / ws
        for b in self.buckets:
            b.handle.wait()
            for p, off in zip(b.params, b.offsets):
                if p.grad is not None:
                    p.grad.copy_(b.flat[off:off + p.numel()].view_as(p.grad)).mul_(inv)
            b.handle = None
            b.pending = len(b.params)


def ensure_process_group():
    """Called by Pix2PixTrainer: the reference's train.py knows nothing about torch.distributed, so when it is launched
    under torchrun (WORLD_SIZE > 1 in the environment) the trainer itself joins the process group -- NCCL, one GPU per
    process (LOCAL_RANK) -- instead of silently running N independent trainings.  Returns (rank, world_size)."""
    import os
    ws_env = int(os.environ.get("WORLD_SIZE", "1"))
    if ws_env > 1 and not (dist.is_available() and dist.is_initialized()):
        if not dist.is_available():
            raise RuntimeError("WORLD_SIZE=%d but torch.distributed is not available" % ws_env)
        if torch.cuda.is_available():
            local = int(os.environ.get("LOCAL_RANK", "0"))
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    if ws_env > 1 and world_size() != ws_env:
        raise RuntimeError("WORLD_SIZE=%d in the environment but the process group has %d ranks" % (ws_env, world_size()))
    return rank(), world_size()


def shard_of(n_items):
    """Index range of this rank's shard of `n_items` samples (a data loader that is not rank-aware feeds every rank the
    same global batch; the trainer can then keep only its own shard)."""
    ws, r = world_size(), rank()
    per = (n_items + ws - 1) // ws
    return range(min(r * per, n_items), min((r + 1) * per, n_items))


def broadcast_module(module, src=0):
    """Make every rank start from rank `src`'s parameters and buffers."""
    if world_size() == 1:
        return
    with torch.no_grad():
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t, src)
