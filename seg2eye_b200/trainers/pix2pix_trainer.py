"""Pix2PixTrainer mirror (reference trainers/pix2pix_trainer.py:9-88).

Data parallelism (beyond the reference, whose README rules multi-GPU training out): launched under torchrun the
trainer joins the NCCL process group itself (the reference's train.py never would), broadcasts rank 0's freshly
initialised / loaded networks so that all replicas start identical, averages the G+E and D gradients across ranks
(seg2eye_b200.parallel) and lets only rank 0 write checkpoints.

`enable_cuda_graphs(example_batch)` captures the generator step and the discriminator step into CUDA graphs, so that a
training iteration is a handful of graph launches instead of ~1300 kernel launches driven from Python:
  * one process: [forward + backward + Adam] is ONE graph per step;
  * several ranks: [forward + backward] and [Adam] are two graphs with the NCCL all-reduce issued eagerly between them
    (with --ada_target also the all-reduce of the D step's sign record; the controller's update is in the [Adam] graph);
    gradients are accumulated straight into the flat all-reduce buckets (parallel.GradReducer.bind_flat_grads), the
    1/world_size factor rides on the loss."""
import torch

from .. import parallel
from ..models.pix2pix_model import Pix2PixModel


class Pix2PixTrainer():
    def __init__(self, opt):
        self.opt = opt
        self.rank, self.world = parallel.ensure_process_group()
        self.pix2pix_model = Pix2PixModel(opt)
        self.pix2pix_model_on_one_gpu = self.pix2pix_model
        self.generated = None
        m = self.pix2pix_model
        if self.world > 1:
            # every replica must start from the same weights AND the same spectral-norm u/v / BatchNorm buffers (both are
            # randomly initialised per process); the EMA nets are rank 0's copies of its G / E or its loaded averages
            for net in (m.netG, m.netD, m.netE, m.netG_ema, m.netE_ema):
                if net is not None:
                    parallel.broadcast_module(net, 0)
            if m.diffaug_state is not None:     # one seed for all ranks: rank r draws for global samples r * B + b
                torch.distributed.broadcast(m.diffaug_state, 0)
            for t in (m.ada_state or {}).values():     # one augmentation probability for all ranks
                torch.distributed.broadcast(t, 0)
            from .. import ops
            ops.bump_weights_epoch()
        if opt.isTrain:
            self.optimizer_G, self.optimizer_D = self.pix2pix_model_on_one_gpu.create_optimizers(opt)
            self.old_lr = opt.lr
            self.reducer_G = parallel.GradReducer(list(m.netG.parameters()) + (list(m.netE.parameters()) if m.netE is not None else []))
            self.reducer_D = parallel.GradReducer(list(m.netD.parameters()))
            if getattr(opt, 'continue_train', False):     # Adam moments / step counts, when a previous run saved them
                from .. import util
                util.load_optimizer(self.optimizer_G, 'G', opt.which_epoch, opt, self._opt_nets('G'))
                util.load_optimizer(self.optimizer_D, 'D', opt.which_epoch, opt, self._opt_nets('D'))
                saved = util.load_optimizer_entry('D', opt.which_epoch, opt, 'diffaug')
                if m.diffaug_state is not None and saved is not None:    # else: the fresh seed, counter 0
                    m.diffaug_state.copy_(torch.tensor([saved['seed'], saved['counter']], dtype=torch.int64))
                    m.load_ada_checkpoint(saved)
        self._graphs = False

    def _opt_nets(self, which):
        m = self.pix2pix_model
        return (('G', m.netG), ('E', m.netE)) if which == 'G' else (('D', m.netD),)

    # ------------------------------------------------------------------ step bodies
    def _ada_allreduce(self, which):
        """--ada_target with several ranks: sum the D step's sign / count record over the ranks (2 num_D + 1 doubles)."""
        m = self.pix2pix_model
        if which == 'D' and m.ada_target > 0 and self.world > 1:
            torch.distributed.all_reduce(m.ada_state['record'])

    def _ada_update(self, which):
        if which == 'D' and self.pix2pix_model.ada_target > 0:
            self.pix2pix_model.ada_update()

    def _fb(self, which, data, scale=1.0):
        """forward + backward of one step; `scale` multiplies the loss that is differentiated (1/world_size when the
        gradients are summed across ranks afterwards), never the reported losses."""
        m = self.pix2pix_model
        if which == 'G':
            losses, generated = m(data, mode='generator')
        else:
            losses, generated = m(data, mode='discriminator'), None
        total = sum(losses.values()).mean()
        (total if scale == 1.0 else total * scale).backward()
        return losses, generated

    def _eager_step(self, which, data):
        opt_, red = (self.optimizer_G, self.reducer_G) if which == 'G' else (self.optimizer_D, self.reducer_D)
        self.reducer_G.armed, self.reducer_D.armed = which == 'G', which == 'D'
        self.pix2pix_model.train()
        opt_.zero_grad()
        losses, generated = self._fb(which, data)
        red.allreduce()
        self._ada_allreduce(which)
        self._ada_update(which)
        opt_.step()
        return losses, generated

    def _split_step(self, which, data):
        """The multi-rank CUDA-graph step executed eagerly (warm-up / capture bodies share this code)."""
        opt_, red = (self.optimizer_G, self.reducer_G) if which == 'G' else (self.optimizer_D, self.reducer_D)
        red.zero_flat()
        out = self._fb(which, data, 1.0 / self.world)
        red.allreduce_flat()
        self._ada_allreduce(which)
        self._ada_update(which)
        opt_.step()
        return out

    # ------------------------------------------------------------------ CUDA-graph fast path
    def enable_cuda_graphs(self, example_data, warmup=3):
        """Capture the G step and the D step for batches shaped like `example_data` (label (B,1,H,W),
        style_image (B,ns,1,H,W), target (B,1,H,W)).  Afterwards run_*_one_step copy the batch into static device
        buffers and replay.  Shapes must not change; call disable_cuda_graphs() to return to eager execution.
        Capture is side-effect free: every piece of state the warm-up iterations touch is restored afterwards.
        Callers that ran eager steps before must not hold on to loss tensors of those steps (anything with a grad_fn):
        they keep the parameters' gradient accumulators bound to the stream of the eager steps, which a capturing stream
        cannot join ("operation would make the legacy stream depend on a capturing blocking stream")."""
        import gc
        from .. import ops
        dev = self.pix2pix_model.device()
        m = self.pix2pix_model
        m.train()
        multi = self.world > 1
        # autograd graphs of earlier eager steps keep the parameters' AccumulateGrad nodes bound to the legacy stream,
        # which cannot be joined from a capturing stream: drop every reference to them before warming up
        for name in ('g_losses', 'd_losses'):
            if getattr(self, name, None) is not None:
                setattr(self, name, {k: v.detach() for k, v in getattr(self, name).items()})
        if self.generated is not None:
            self.generated = self.generated.detach()
        m.reset_loss_log()
        gc.collect()
        self._static = {'label': example_data['label'].long().to(dev).clone(),
                        'target': example_data['target'].float().to(dev).clone()}
        if 'style_image' in example_data:
            self._static['style_image'] = example_data['style_image'].float().to(dev).clone()
        m.sync_ema()
        tensors = [t for net in (m.netG, m.netD, m.netE, m.netG_ema, m.netE_ema) if net is not None
                   for t in list(net.parameters()) + list(net.buffers())]
        if m.diffaug_state is not None:     # the warm-up steps draw: the counter is restored with the weights
            tensors.append(m.diffaug_state)
        tensors += list((m.ada_state or {}).values())     # ... and they move the augmentation probability
        opts = (self.optimizer_G, self.optimizer_D)
        if multi:     # the capture set-up below runs on a side stream: no all-reduce launches from inside backward there
            self.reducer_G.remove_hooks()
            self.reducer_D.remove_hooks()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):   # one throw-away iteration so that optimizer state (and the buckets) exist
            for o in opts:
                o.zero_grad(set_to_none=True)
            if len(self.optimizer_G.state) == 0 or (multi and self.reducer_G.buckets is None):
                snap0 = [t.detach().clone() for t in tensors]
                fresh = len(self.optimizer_G.state) == 0
                self._eager_step('G', dict(self._static))
                self._eager_step('D', dict(self._static))
                if fresh:
                    self.reset_optimizers()
                for t, s0 in zip(tensors, snap0):
                    t.detach().copy_(s0)
            if multi:
                self.reducer_G.bind_flat_grads()
                self.reducer_D.bind_flat_grads()
        torch.cuda.current_stream().wait_stream(side)
        opt_tensors = [st[k] for o in opts for st in o.state.values() for k in ('exp_avg', 'exp_avg_sq')]
        opt_tensors += [g['_s2e_state'] for o in opts for g in o.param_groups if g.get('_s2e_state') is not None]
        snap = [t.detach().clone() for t in tensors + opt_tensors]

        def step(which):
            if multi:
                return self._split_step(which, dict(self._static))
            (self.optimizer_G if which == 'G' else self.optimizer_D).zero_grad(set_to_none=True)
            out = self._fb(which, dict(self._static))
            self._ada_update(which)
            (self.optimizer_G if which == 'G' else self.optimizer_D).step()
            return out

        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):     # fills the packed-weight cache, sets function attributes, warms the allocator
                step('G')
                step('D')
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()    # the graphs allocate from a private pool; give the eager cache back first
        self._gr = {}
        pool = None
        for which in ('G', 'D'):
            opt_, red = (self.optimizer_G, self.reducer_G) if which == 'G' else (self.optimizer_D, self.reducer_D)
            m.reset_loss_log()
            g_fb = torch.cuda.CUDAGraph()
            if multi:
                with torch.cuda.graph(g_fb, pool=pool):
                    red.zero_flat()
                    out = self._fb(which, dict(self._static), 1.0 / self.world)
                pool = g_fb.pool()
                red.allreduce_flat()
                self._ada_allreduce(which)
                g_opt = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_opt, pool=pool):
                    self._ada_update(which)
                    opt_.step()
            else:
                opt_.zero_grad(set_to_none=True)
                with torch.cuda.graph(g_fb, pool=pool):
                    out = self._fb(which, dict(self._static))
                    self._ada_update(which)
                    opt_.step()
                pool = g_fb.pool()
                g_opt = None
            # raw-loss tensors the model logged during the capture (L1/raw ...): static outputs of the graph, re-logged
            # after every replay (the reference's train.py prints them)
            log = {k: list(v) for k, v in m.loss_log.items()}
            self._gr[which] = (g_fb, g_opt, out, log)
        m.reset_loss_log()
        for t, s0 in zip(tensors + opt_tensors, snap):
            t.detach().copy_(s0)
        ops.bump_weights_epoch()
        ops.repack_stale()   # the graphs re-pack after their own Adam; the restored weights need it once, here
        self._graphs = True

    def reset_optimizers(self):
        """Both optimizers as freshly constructed: zero Adam moments and step counts, and the EMA nets copies of G / E,
        written in place so that captured CUDA graphs keep reading the same tensors."""
        self.pix2pix_model.reset_ema()
        for o in (self.optimizer_G, self.optimizer_D):
            for st in o.state.values():
                st['exp_avg'].zero_()
                st['exp_avg_sq'].zero_()
            for g in o.param_groups:
                if g.get('_s2e_state') is not None:
                    g['_s2e_state'][0].zero_()

    def disable_cuda_graphs(self):
        self._graphs = False
        self._gr = None
        for red, opt_ in ((self.reducer_G, self.optimizer_G), (self.reducer_D, self.optimizer_D)):
            if red.flat_bound:
                red.unbind_flat_grads()
            opt_.zero_grad(set_to_none=True)

    def _load_static(self, data):
        for k, buf in self._static.items():
            src = data[k]
            if src.shape != buf.shape:
                raise RuntimeError("CUDA-graph step captured for %s %s, got %s" % (k, tuple(buf.shape), tuple(src.shape)))
            if src.data_ptr() != buf.data_ptr():
                buf.copy_(src, non_blocking=True)
        data.update(self._static)   # the reference mutates `data` in place too (pix2pix_model.py:140-158)

    def _replay(self, which, data):
        """NOTE: the returned losses / image are the graph's static output buffers -- the next replay overwrites them
        (clone what must outlive the step)."""
        from .. import ops
        if ops.repack_pending():     # weights changed behind the graphs' back (load_network, manual edits)
            ops.repack_stale()
        self._load_static(data)
        g_fb, g_opt, out, log = self._gr[which]
        g_fb.replay()
        if g_opt is not None:
            (self.reducer_G if which == 'G' else self.reducer_D).allreduce_flat()
            self._ada_allreduce(which)
            g_opt.replay()
        if which == 'G':
            self.optimizer_G.ema_written()
        for k, vals in log.items():
            for v in vals:
                self.pix2pix_model.add_to_loss_log(k, v.clone())
        return out

    # ------------------------------------------------------------------ reference API
    def run_generator_one_step(self, data):
        self.pix2pix_model.sync_ema()
        if self._graphs:
            self.g_losses, self.generated = self._replay('G', data)
        else:
            self.g_losses, self.generated = self._eager_step('G', data)

    def run_discriminator_one_step(self, data):
        if self._graphs:
            self.d_losses = self._replay('D', data)[0]
        else:
            self.d_losses = self._eager_step('D', data)[0]

    def get_latest_losses(self, include_log_losses=False):
        losses = {**self.g_losses, **self.d_losses}
        if include_log_losses:
            losses = {**losses, **self.pix2pix_model_on_one_gpu.get_loss_log()}
            self.pix2pix_model_on_one_gpu.reset_loss_log()
        return losses

    def get_latest_generated(self):
        return self.generated

    def save(self, epoch):
        if self.rank == 0:      # replicas are identical; concurrent writers of the same file would corrupt it
            self.pix2pix_model_on_one_gpu.save(epoch)
            if self.opt.isTrain:
                from .. import util
                util.save_optimizer(self.optimizer_G, 'G', epoch, self.opt, self._opt_nets('G'))
                st = self.pix2pix_model.diffaug_state
                extra = None
                if st is not None:
                    extra = {'diffaug': dict(seed=int(st[0]), counter=int(st[1]), **self.pix2pix_model.ada_checkpoint())}
                util.save_optimizer(self.optimizer_D, 'D', epoch, self.opt, self._opt_nets('D'), extra)
        if self.world > 1:
            torch.distributed.barrier()

    def update_learning_rate(self, epoch):
        """Linear decay (pix2pix_trainer.py:68-88): constant for the first `niter` epochs, then lr/niter_decay is taken
        off once per epoch; under TTUR the generator runs at half and the discriminator at twice the nominal rate."""
        if epoch <= self.opt.niter:
            return
        new_lr = self.old_lr - self.opt.lr / self.opt.niter_decay
        if new_lr == self.old_lr:
            return
        g_scale, d_scale = (1.0, 1.0) if self.opt.no_TTUR else (0.5, 2.0)
        for optimizer, scale in ((self.optimizer_G, g_scale), (self.optimizer_D, d_scale)):
            for group in optimizer.param_groups:
                group['lr'] = new_lr * scale
            optimizer.sync_hyperparams()
        print('update learning rate: %f -> %f' % (self.old_lr, new_lr))
        self.old_lr = new_lr
