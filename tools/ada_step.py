"""Cost of the per-sample gates and of ADA (`--diff_augment_p`, `--ada_target`) on one GPU: ms/step of the CUDA-graph
training step (c2, R2, B16) with the full DiffAugment policy at p = 1 (today's path) and with ADA on and p held near 0.5
(a start value of 0.5 and an --ada_kimg so large that p does not move), alternated in one process; and every new launch
timed on its own with CUDA events against the launch it replaces, at the step's shapes.

    python tools/ada_step.py [--steps 20] [--rounds 3] [--iters 200] [--policy color,translation,cutout]
"""
import argparse
import contextlib
import io
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--policy", default="color,translation,cutout")
    args = ap.parse_args()
    import bench
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import _lib as L
    from seg2eye_b200 import ops

    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer

    if not torch.cuda.is_available():
        raise SystemExit("ada_step.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    res, batch = "R2", 16
    trainers, data = {}, None
    for name, extra in (("p=1", {}), ("ada p~0.5", dict(ada_target=0.6, diff_augment_p=0.5, ada_kimg=1e12))):
        oopt, opt = bench.make_opts(res, batch, "c2")
        opt.diff_augment = args.policy
        for k, v in extra.items():
            setattr(opt, k, v)
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
    p_end = float(trainers["ada p~0.5"].pix2pix_model.ada_state["p"])

    # the launches alone, at the step's shapes
    B, H, W = batch, data["label"].shape[-2], data["label"].shape[-1]
    nc = oopt.label_nc
    cpad = -(-(nc + 1) // 16) * 16
    seg = torch.rand(B, nc, H, W, device="cuda")
    fake, real = torch.rand(B, 1, H, W, device="cuda"), torch.rand(B, 1, H, W, device="cuda")
    out = torch.empty(2 * B, H, W, cpad, dtype=torch.bfloat16, device="cuda")
    dout = torch.randn(2 * B, H, W, cpad, device="cuda").to(torch.bfloat16)
    dfake = torch.empty(B, 1, H, W, device="cuda")
    state = torch.tensor([7, 0], dtype=torch.int64, device="cuda")
    p = torch.tensor([0.5], dtype=torch.float64, device="cuda")
    rec, mask = ops.diffaug_draw_p(state, p, B, 0, H, W)
    means = torch.empty(2 * B, device="cuda")
    L.call("s2e_diffaug_means", L.ptr(fake), L.ptr(real), B, H, W, L.ptr(means), L.stream())
    scratch = torch.empty(B, dtype=torch.float64, device="cuda")
    _, bits = ops.parse_diff_augment(args.policy)
    # the scale-0 logit head of D at R2: 512 -> 1 channel, 4x4, stride 1, pad 2, on the 2B x 81 x 49 map
    cfg = ops.ConvCfg(4, 4, 1, 2, L.ACT_NONE)
    Hi, Wi = H // 8 + 1, W // 8 + 1
    Ho, Wo = ops.conv_out_hw(cfg, Hi, Wi)
    taps = ops.conv_taps(cfg)
    D = torch.randn(2 * B * Hi * Wi, 16, device="cuda")
    y = torch.empty(2 * B, Ho, Wo, 1, dtype=torch.bfloat16, device="cuda")
    desc = ops._desc(2 * B, Hi, Wi, 512, Ho, Wo, 1, taps, L.ACT_NONE)
    sums = torch.zeros(7, device="cuda")
    sgn = torch.zeros(1, device="cuda")
    ada = {"p": torch.tensor([0.5], dtype=torch.float64, device="cuda"), "acc": torch.zeros(6, dtype=torch.float64, device="cuda"),
           "pos": torch.zeros(1, dtype=torch.int32, device="cuda"),
           "record": torch.tensor([1.0, 2.0, 1.0, 2.0, 16.0], dtype=torch.float64, device="cuda")}
    s = L.stream()
    P = L.ptr
    launch = {
        "s2e_diffaug_draw": lambda: L.call("s2e_diffaug_draw", P(state), B, 0, H, W, P(rec), s),
        "s2e_diffaug_draw_p": lambda: L.call("s2e_diffaug_draw_p", P(state), P(p), B, 0, H, W, P(rec), P(mask), s),
        "s2e_make_d_input_aug": lambda: L.call("s2e_make_d_input_aug", P(seg), P(fake), P(real), B, nc, H, W, cpad, P(rec),
                                               P(means), bits, P(out), s),
        "s2e_make_d_input_aug_masked": lambda: L.call("s2e_make_d_input_aug_masked", P(seg), P(fake), P(real), B, nc, H, W, cpad,
                                                      P(rec), P(means), bits, P(mask), P(out), s),
        "s2e_d_input_grad_aug": lambda: L.call("s2e_d_input_grad_aug", P(dout), B, nc, H, W, cpad, P(rec), bits, P(scratch),
                                               P(dfake), s),
        "s2e_d_input_grad_aug_masked": lambda: L.call("s2e_d_input_grad_aug_masked", P(dout), B, nc, H, W, cpad, P(rec), bits,
                                                      P(mask), P(scratch), P(dfake), s),
        "s2e_head_gather": lambda: L.call("s2e_head_gather", desc, P(D), None, None, P(y), P(sums), s),
        "s2e_head_gather_signs": lambda: L.call("s2e_head_gather_signs", desc, P(D), None, None, P(y), P(sums), P(sums[6:]), s),
        "s2e_reduce_loss SIGN": lambda: L.call("s2e_reduce_loss", P(y[B:]), None, B * Ho * Wo, 0, L.RED_SIGN, 1.0, 0.0, P(sgn), 0, s),
        "s2e_ada_update": lambda: ops.ada_update(ada, 0.6, 1e12, 4),
    }
    ms = {k: [] for k in launch}
    for f in launch.values():
        f()
    for _ in range(args.rounds):
        for k, f in launch.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                f()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.iters)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print("card: %s; workload c2, %s, B%d, N = 1, CUDA graphs, policy %s, %d rounds x %d steps alternated"
          % (q, res, batch, args.policy, args.rounds, args.steps))
    for name, ts in times.items():
        print("%-12s ms/step %s  best %.3f  images/s %.1f" % (name, " ".join("%.3f" % v for v in ts), min(ts),
                                                              batch / (min(ts) / 1e3)))
    off, on = (min(v) for v in times.values())
    print("ADA step overhead: %+.3f ms/step (%+.2f%%); p at the end of the ADA run: %.6f" % (on - off, 100 * (on / off - 1), p_end))
    print("launches at B%d, %dx%d, nc %d, Cpad %d, p = 0.5 masks; logit head 2B x %dx%d; %d launches per timing window:"
          % (B, H, W, nc, cpad, Ho, Wo, args.iters))
    for k, ts in ms.items():
        print("%-28s ms %s  best %.4f" % (k, " ".join("%.4f" % v for v in ts), min(ts)))
    best = {k: min(v) for k, v in ms.items()}
    g = sum(best[k + "_masked"] - best[k] for k in ("s2e_make_d_input_aug", "s2e_d_input_grad_aug")) + \
        best["s2e_diffaug_draw_p"] - best["s2e_diffaug_draw"]
    d = best["s2e_make_d_input_aug_masked"] - best["s2e_make_d_input_aug"] + best["s2e_diffaug_draw_p"] - best["s2e_diffaug_draw"] + \
        2 * (best["s2e_head_gather_signs"] - best["s2e_head_gather"]) + best["s2e_ada_update"]
    print("launch time added per G step %+.4f ms, per D step %+.4f ms (two logit heads, one controller launch)" % (g, d))


if __name__ == "__main__":
    main()
