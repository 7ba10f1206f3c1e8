"""Cost of `--diff_augment xflip,geometric` on one GPU: ms/step of the CUDA-graph training step (c2, R2, B16) with all
five ops at p = 0.5 against the three DiffAugment ops at p = 0.5 (today's gated path), alternated in one process; and the
draw, the layout kernel and its adjoint timed on their own with CUDA events against the launches they replace, at the
step's shapes.  The adjoint's gather is also timed with every sample forced to the strongest zoom-out the draw can produce
(s and a at their bound 2^(-0.2 * 5.9), so that many mirror images of each source pixel are reachable).

    python tools/geomaug_step.py [--steps 20] [--rounds 3] [--iters 200]
"""
import argparse
import contextlib
import io
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

THREE = "color,translation,cutout"
FIVE = "color,xflip,geometric,translation,cutout"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    import bench
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import _lib as L
    from seg2eye_b200 import ops
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer

    if not torch.cuda.is_available():
        raise SystemExit("geomaug_step.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    res, batch = "R2", 16
    trainers, data = {}, None
    for name, policy in (("3 ops p=0.5", THREE), ("5 ops p=0.5", FIVE)):
        oopt, opt = bench.make_opts(res, batch, "c2")
        opt.diff_augment, opt.diff_augment_p = policy, 0.5
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
    rec, geom, mask = ops.diffaug_draw_geom(state, p, B, 0, H, W)
    means = torch.empty(2 * B, device="cuda")
    L.call("s2e_diffaug_means", L.ptr(fake), L.ptr(real), B, H, W, L.ptr(means), L.stream())
    scratch = torch.empty(B, dtype=torch.float64, device="cuda")
    bits3, bits5 = ops.parse_diff_augment(THREE)[1], ops.parse_diff_augment(FIVE)[1]
    z = 2.0 ** (0.2 * 5.9)     # the strongest zoom-out: 1/s = 1/a = z, rotated by 0.3 rad, with a fractional shift
    c, s_ = math.cos(0.3), math.sin(0.3)
    zoom = torch.tensor([z * z * c, s_, 0.1 * W, -z * z * s_, c, -0.05 * H, 0, 0], dtype=torch.float32,
                        device="cuda").repeat(B, 1)
    mask_zoom = mask | L.DIFFAUG_GEOMETRIC
    s = L.stream()
    P = L.ptr
    launch = {
        "s2e_diffaug_draw_p": lambda: L.call("s2e_diffaug_draw_p", P(state), P(p), B, 0, H, W, P(rec), P(mask), s),
        "s2e_diffaug_draw_geom": lambda: L.call("s2e_diffaug_draw_geom", P(state), P(p), B, 0, H, W, P(rec), P(geom), P(mask), s),
        "s2e_make_d_input_aug_masked": lambda: L.call("s2e_make_d_input_aug_masked", P(seg), P(fake), P(real), B, nc, H, W, cpad,
                                                      P(rec), P(means), bits3, P(mask), P(out), s),
        "s2e_make_d_input_aug_geom": lambda: L.call("s2e_make_d_input_aug_geom", P(seg), P(fake), P(real), B, nc, H, W, cpad,
                                                    P(rec), P(means), bits5, P(mask), P(geom), P(out), s),
        "s2e_d_input_grad_aug_masked": lambda: L.call("s2e_d_input_grad_aug_masked", P(dout), B, nc, H, W, cpad, P(rec), bits3,
                                                      P(mask), P(scratch), P(dfake), s),
        "s2e_d_input_grad_aug_geom": lambda: L.call("s2e_d_input_grad_aug_geom", P(dout), B, nc, H, W, cpad, P(rec), bits5,
                                                    P(mask), P(geom), P(scratch), P(dfake), s),
        "s2e_d_input_grad_aug_geom zoom-out": lambda: L.call("s2e_d_input_grad_aug_geom", P(dout), B, nc, H, W, cpad, P(rec),
                                                             bits5, P(mask_zoom), P(zoom), P(scratch), P(dfake), s),
    }
    # the draws above advanced the counter; the timed windows redraw in place, so the masks stay at p = 0.5 throughout
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
    print("card: %s; workload c2, %s, B%d, N = 1, CUDA graphs, p = 0.5, %d rounds x %d steps alternated"
          % (q, res, batch, args.rounds, args.steps))
    for name, ts in times.items():
        print("%-12s ms/step %s  best %.3f  images/s %.1f" % (name, " ".join("%.3f" % v for v in ts), min(ts),
                                                              batch / (min(ts) / 1e3)))
    off, on = (min(v) for v in times.values())
    print("xflip + geometric step overhead: %+.3f ms/step (%+.2f%%)" % (on - off, 100 * (on / off - 1)))
    print("launches at B%d, %dx%d, nc %d, Cpad %d, p = 0.5; %d launches per timing window:" % (B, H, W, nc, cpad, args.iters))
    for k, ts in ms.items():
        print("%-36s ms %s  best %.4f" % (k, " ".join("%.4f" % v for v in ts), min(ts)))
    best = {k: min(v) for k, v in ms.items()}
    g = sum(best[k + "_geom"] - best[k + "_masked"] for k in ("s2e_make_d_input_aug", "s2e_d_input_grad_aug")) + \
        best["s2e_diffaug_draw_geom"] - best["s2e_diffaug_draw_p"]
    d = best["s2e_make_d_input_aug_geom"] - best["s2e_make_d_input_aug_masked"] + best["s2e_diffaug_draw_geom"] - \
        best["s2e_diffaug_draw_p"]
    print("launch time added per G step %+.4f ms, per D step %+.4f ms" % (g, d))


if __name__ == "__main__":
    main()
