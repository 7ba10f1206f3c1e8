"""Run-to-run reproducibility of the bench training trajectory: two trainers built from the same seed train on the same
batch through the CUDA-graph path (bench.py's c2 workload, R2, batch 16); prints how far their generated images and
losses are apart after a given number of steps.  The weight-gradient and loss reductions add with float atomics, so
step 1 agrees to rounding only, and Adam(beta1 = 0) from the small initial weights amplifies that from step 2 on.

    python tools/trajectory_repro.py > profiles/rXX_trajectory_repro.txt"""
import contextlib
import io
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

import bench  # noqa: E402
from oracle import seg2eye_oracle as O  # noqa: E402
from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer  # noqa: E402

REPORT = (1, 2, 5, 10, 20, 50)


def trajectory():
    oopt, opt = bench.make_opts("R2", 16, "c2")
    opt.gpu_ids = [0]
    torch.manual_seed(1234)
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    dev = {k: v.cuda() for k, v in O.synth_batch(oopt, 16, 1234).items()}
    tr.enable_cuda_graphs(dev, warmup=1)
    out = {}
    for s in range(1, max(REPORT) + 1):
        tr.run_generator_one_step(dict(dev))
        tr.run_discriminator_one_step(dict(dev))
        if s in REPORT:
            out[s] = (tr.get_latest_generated().detach().clone(),
                      {k: float(v.reshape(-1)[0]) for k, v in tr.get_latest_losses().items()})
    return out


def main():
    torch.cuda.set_device(0)
    print(subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
    a = trajectory()
    torch.cuda.empty_cache()
    b = trajectory()
    print("step  image_rel_l2  max_loss_rel  losses_rel")
    for s in REPORT:
        (ia, la), (ib, lb) = a[s], b[s]
        rel = {k: abs(la[k] - lb[k]) / max(abs(lb[k]), 1e-12) for k in la}
        print("%4d  %12.3g  %12.3g  %s" % (s, float((ia - ib).norm() / ib.norm()), max(rel.values()),
                                           " ".join("%s=%.2g" % kv for kv in rel.items())), flush=True)


if __name__ == "__main__":
    main()
