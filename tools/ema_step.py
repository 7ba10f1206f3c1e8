"""Cost of `--ema_decay` on one GPU: ms/step of the CUDA-graph training step (c2, R2, B16) with the EMA off and on,
alternated in one process, and the G optimizer's Adam launches timed on their own with CUDA events, s2e_adam_multi
against s2e_adam_multi_ema, over the real G+E parameters.

    python tools/ema_step.py [--steps 20] [--rounds 3] [--adam-iters 500] [--ema-decay 0.999]
"""
import argparse
import contextlib
import ctypes as C
import io
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def adam_args(opt_, ema):
    """The C-ABI arguments optim.Adam.step passes for the G group (its grads are the captured graph's static buffers), on
    a copy of the group's device state; the caller keeps that copy (last return value) alive while it launches."""
    from seg2eye_b200 import _lib as L
    group = opt_.param_groups[0]
    ps = [p for p in group['params'] if p.grad is not None]
    n = len(ps)
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    st = group['_s2e_state'].clone()
    b1, b2 = group['betas']
    args = (n, arr(ps), arr([p.grad for p in ps]), arr([opt_.state[p]['exp_avg'] for p in ps]),
            arr([opt_.state[p]['exp_avg_sq'] for p in ps]), (C.c_longlong * n)(*[p.numel() for p in ps]), L.ptr(st), b1, b2,
            group['eps'], group['weight_decay'])
    return args, (arr([ema[p] for p in ps]) if ema else None), sum(p.numel() for p in ps), st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--adam-iters", type=int, default=500)
    ap.add_argument("--ema-decay", type=float, default=0.999)
    args = ap.parse_args()
    import bench
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import _lib as L
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer

    if not torch.cuda.is_available():
        raise SystemExit("ema_step.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    res, batch = "R2", 16
    trainers, data = {}, None
    for name, beta in (("ema off", 0.0), ("ema %g" % args.ema_decay, args.ema_decay)):
        oopt, opt = bench.make_opts(res, batch, "c2")
        opt.ema_decay = beta
        torch.manual_seed(1234)
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        if data is None:
            data = {k: v.cuda() for k, v in O.synth_batch(oopt, batch, 1234).items()}
        tr.enable_cuda_graphs(data, warmup=1)
        trainers[name] = tr

    times = {k: [] for k in trainers}
    for _ in range(args.rounds):
        for name, tr in trainers.items():
            for _ in range(3):
                tr.run_generator_one_step(dict(data))
                tr.run_discriminator_one_step(dict(data))
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                tr.run_generator_one_step(dict(data))
                tr.run_discriminator_one_step(dict(data))
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)

    # the Adam launches alone, on the EMA trainer's G group (the weights move; nothing runs after this)
    tr = trainers["ema %g" % args.ema_decay]
    base, ema_ptrs, n_params, _state = adam_args(tr.optimizer_G, tr.optimizer_G.ema)   # _state: keeps the device state alive
    s = L.stream()
    launch = {"s2e_adam_multi": lambda: L.call("s2e_adam_multi", *base, s),
              "s2e_adam_multi_ema": lambda: L.call("s2e_adam_multi_ema", *base, ema_ptrs, args.ema_decay, s)}
    adam_ms = {k: [] for k in launch}
    for f in launch.values():
        f()
    for _ in range(args.rounds):
        for k, f in launch.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.adam_iters):
                f()
            e1.record()
            torch.cuda.synchronize()
            adam_ms[k].append(e0.elapsed_time(e1) / args.adam_iters)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print("card: %s; workload c2, %s, B%d, N = 1, CUDA graphs, %d rounds x %d steps alternated"
          % (q, res, batch, args.rounds, args.steps))
    for name, ts in times.items():
        print("%-10s ms/step %s  best %.3f  images/s %.1f" % (name, " ".join("%.3f" % v for v in ts), min(ts),
                                                              batch / (min(ts) / 1e3)))
    off, on = (min(v) for v in times.values())
    print("EMA step overhead: %+.3f ms/step (%+.2f%%)" % (on - off, 100 * (on / off - 1)))
    print("Adam launches over %d G+E parameters, %d launches per timing window:" % (n_params, args.adam_iters))
    for k, ts in adam_ms.items():
        nbytes = n_params * (28 if k == "s2e_adam_multi" else 36)     # p g m v read, p m v written (+ e read and written)
        print("%-20s ms %s  best %.3f  %.0f GB/s (%d B/param)" % (k, " ".join("%.3f" % v for v in ts), min(ts),
                                                                 nbytes / (min(ts) / 1e3) / 1e9, nbytes // n_params))
    a, b = (min(v) for v in adam_ms.values())
    print("EMA Adam overhead: %+.3f ms per G step" % (b - a))


if __name__ == "__main__":
    main()
