"""ms/step and images/s of `--norm_G spectralspadebatch3x3` against `spectralspadesyncbatch3x3` (SyncBatchNorm in every
SPADE layer), CUDA-graph mode, the two configurations alternated within one process group.  Also counts the
collectives that the shared statistics issue per G step and per D step (one eager step each).  Run under
torch.distributed.run, one process per GPU:

    python -m torch.distributed.run --nproc-per-node N tools/syncbn_step.py [--workload c2|c5] [--steps 20] [--rounds 3]
"""
import argparse
import contextlib
import io
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2", choices=("c2", "c5"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import bench
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import ops
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res, batch = {"c2": ("R2", 16), "c5": ("S256", 16)}[args.workload]
    trainers, data = {}, None
    for norm in ("spectralspadebatch3x3", "spectralspadesyncbatch3x3"):
        oopt, opt = bench.make_opts(res, batch, args.workload)
        opt.norm_G = oopt.norm_G = norm
        opt.gpu_ids = [local]
        torch.manual_seed(1234 + rank)
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Pix2PixTrainer(opt)
        if data is None:
            host = O.synth_batch(oopt, batch, 1234 + rank)
            if tr.pix2pix_model.netE is None:
                host.pop("style_image")
            data = {k: v.cuda() for k, v in host.items()}
        counts = {}
        for which in ("G", "D"):       # one eager step each: collectives issued by the shared statistics
            n0 = ops._state.get("sync_collectives", 0)
            (tr.run_generator_one_step if which == "G" else tr.run_discriminator_one_step)(dict(data))
            counts[which] = ops._state.get("sync_collectives", 0) - n0
        tr.enable_cuda_graphs(data, warmup=1)
        trainers[norm] = (tr, counts)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    times = {k: [] for k in trainers}
    for _ in range(args.rounds):
        for norm, (tr, _) in trainers.items():
            for _ in range(3):
                tr.run_generator_one_step(dict(data))
                tr.run_discriminator_one_step(dict(data))
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                tr.run_generator_one_step(dict(data))
                tr.run_discriminator_one_step(dict(data))
            e1.record()
            sync()
            t = torch.tensor([e0.elapsed_time(e1) / args.steps], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times[norm].append(float(t))
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                           capture_output=True, text=True).stdout.strip()
        print("card: %s; workload %s, %s, B%d per GPU, N = %d, CUDA graphs, %d rounds x %d steps alternated"
              % (q, args.workload, res, batch, world, args.rounds, args.steps))
        for norm, ts in times.items():
            ms = min(ts)
            print("%-28s ms/step %s  best %.2f  images/s %.1f  sync collectives: G step %d, D step %d"
                  % (norm, " ".join("%.2f" % v for v in ts), ms, batch * world / (ms / 1e3), trainers[norm][1]["G"],
                     trainers[norm][1]["D"]))
        b, s = (min(times[k]) for k in trainers)
        print("syncbatch overhead: %+.2f%%" % (100 * (s / b - 1)))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
