"""Cost of `--diff_augment` on one GPU: ms/step of the CUDA-graph training step (c2, R2, B16) with the policy off and with
color,translation,cutout, alternated in one process, and the D-input launches timed on their own with CUDA events, today's
against the augmented ones, at the step's shapes.

    python tools/diffaug_step.py [--steps 20] [--rounds 3] [--iters 200] [--policy color,translation,cutout]
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
        raise SystemExit("diffaug_step.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    res, batch = "R2", 16
    trainers, data = {}, None
    for name, policy in (("off", ""), (args.policy, args.policy)):
        oopt, opt = bench.make_opts(res, batch, "c2")
        opt.diff_augment = policy
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

    # the D-input launches alone, at the step's shapes (seg one-hot NCHW fp32, fake / real fp32, Cpad 16)
    B, H, W = batch, data["label"].shape[-2], data["label"].shape[-1]
    nc = oopt.label_nc
    cpad = -(-(nc + 1) // 16) * 16
    seg = torch.rand(B, nc, H, W, device="cuda")
    fake, real = torch.rand(B, 1, H, W, device="cuda"), torch.rand(B, 1, H, W, device="cuda")
    out = torch.empty(2 * B, H, W, cpad, dtype=torch.bfloat16, device="cuda")
    dout = torch.randn(2 * B, H, W, cpad, device="cuda").to(torch.bfloat16)
    dfake = torch.empty(B, 1, H, W, device="cuda")
    state = torch.tensor([7, 0], dtype=torch.int64, device="cuda")
    rec = ops.diffaug_draw(state, B, 0, H, W)
    means = torch.empty(2 * B, device="cuda")
    scratch = torch.empty(B, dtype=torch.float64, device="cuda")
    _, bits = ops.parse_diff_augment(args.policy)
    s = L.stream()
    P = L.ptr
    launch = {
        "s2e_make_d_input": lambda: L.call("s2e_make_d_input", P(seg), P(fake), P(real), B, nc, H, W, cpad, P(out), s),
        "s2e_d_input_grad": lambda: L.call("s2e_d_input_grad", P(dout), B, nc, H, W, cpad, P(dfake), s),
        "s2e_diffaug_draw": lambda: L.call("s2e_diffaug_draw", P(state), B, 0, H, W, P(rec), s),
        "s2e_diffaug_means": lambda: L.call("s2e_diffaug_means", P(fake), P(real), B, H, W, P(means), s),
        "s2e_make_d_input_aug": lambda: L.call("s2e_make_d_input_aug", P(seg), P(fake), P(real), B, nc, H, W, cpad, P(rec),
                                               P(means), bits, P(out), s),
        "s2e_d_input_grad_aug": lambda: L.call("s2e_d_input_grad_aug", P(dout), B, nc, H, W, cpad, P(rec), bits, P(scratch),
                                               P(dfake), s),
    }
    # bytes moved: fp32 seg + image in, bf16 D input out; one bf16 channel (a 32-byte sector per pixel) in, fp32 out
    in_bytes, d_bytes = 2 * B * H * W * (nc + 1) * 4, 2 * B * H * W * cpad * 2
    nbytes = {"s2e_make_d_input": in_bytes + d_bytes, "s2e_make_d_input_aug": in_bytes + d_bytes,
              "s2e_d_input_grad": B * H * W * (32 + 4), "s2e_d_input_grad_aug": B * H * W * (32 + 4) * (2 if bits & 1 else 1),
              "s2e_diffaug_means": 2 * B * H * W * 4, "s2e_diffaug_draw": B * 24}
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
    print("card: %s; workload c2, %s, B%d, N = 1, CUDA graphs, %d rounds x %d steps alternated"
          % (q, res, batch, args.rounds, args.steps))
    for name, ts in times.items():
        print("%-24s ms/step %s  best %.3f  images/s %.1f" % (name, " ".join("%.3f" % v for v in ts), min(ts),
                                                              batch / (min(ts) / 1e3)))
    off, on = (min(v) for v in times.values())
    print("augmentation step overhead: %+.3f ms/step (%+.2f%%)" % (on - off, 100 * (on / off - 1)))
    print("D-input launches at B%d, %dx%d, nc %d, Cpad %d (policy %s), %d launches per timing window:"
          % (B, H, W, nc, cpad, args.policy, args.iters))
    for k, ts in ms.items():
        print("%-22s ms %s  best %.4f  %.0f GB/s" % (k, " ".join("%.4f" % v for v in ts), min(ts),
                                                   nbytes[k] / (min(ts) / 1e3) / 1e9))
    best = {k: min(v) for k, v in ms.items()}
    g_new = best["s2e_diffaug_draw"] + best["s2e_diffaug_means"] * bool(bits & 1) + best["s2e_make_d_input_aug"] + \
        best["s2e_d_input_grad_aug"]
    g_old = best["s2e_make_d_input"] + best["s2e_d_input_grad"]
    d_new = best["s2e_diffaug_draw"] + best["s2e_diffaug_means"] * bool(bits & 1) + best["s2e_make_d_input_aug"]
    print("per G step: %.4f -> %.4f ms (%+.4f); per D step: %.4f -> %.4f ms (%+.4f)"
          % (g_old, g_new, g_new - g_old, best["s2e_make_d_input"], d_new, d_new - best["s2e_make_d_input"]))


if __name__ == "__main__":
    main()
