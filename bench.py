"""Benchmark of the Seg2Eye SPADE+Style G+D training step (BASELINE.json metric: G+D train images/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--res R1|R2] [--batch B] [--dump-outputs DIR]

One "step" = one Pix2PixTrainer.run_generator_one_step + run_discriminator_one_step over one synthetic batch
(labels: eye-shaped 4-class ellipses; images/targets U(-1,1); reference-initialised weights).  Prints ONE JSON line.

`value`    : whole-job images/s with the batch already resident in HBM when the timed region starts.
`e2e`      : the same metric through the public trainer API fed with pinned HOST tensors each step (H2D of labels,
             style images and target inside the timed region, D2H read of the five loss scalars).
`roofline` : tcgen05 tap-convolution kernels -- algorithmic FLOPs (2*M*N*K per launch, fwd / dgrad / wgrad) over their
             CUDA-event durations inside the timed region, against the measured bf16 GEMM peak.
`cpu_baseline` / --impl reference: the oracle port (plain fp32 PyTorch restatement of the reference, the reference
             itself is Python and does not travel to the GPU box) timed on the host cores on a bounded sample.
--dump-outputs DIR: writes what one step of the timed path returns to a caller as DIR/<name>.npy (float32): the generated
             image and the losses of a training step, the integer images of a c4 sweep.  A training step is dumped from
             the seeded initial weights: after the timed steps they are restored, with a fresh optimizer, and the timed
             path (the same CUDA graphs, the same batch) runs one more step.  Inputs and weights are seeded, so two builds
             of the project run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import torch  # noqa: E402

RES = {"R1": (256, 0.8), "R2": (384, 0.6), "S256": (256, 1.0)}   # crop_size, aspect_ratio -> 320x256 / 640x384 / 256x256 (SURVEY fact 4)
STEP_TFLOP = {"R1": 1.54, "R2": 4.53}        # reference-equivalent FLOPs per image (BASELINE.md section 3)
WORKLOADS = {
    "c2": "Seg2Eye full G+D training step (SPADEStyle G, multiscale PatchGAN D, GAN+feat-match+L1)",
    "c4": "Style-encoder + generator inference sweep (encode 2 style sets, 64-step style interpolation, batch-64 inference, "
          "device tail to 640x400 integers)",
    "c5": "Original SPADE generator (no style branch), 35-class segmap, full G+D training step (multiscale PatchGAN D, GAN+feat-match+L1)",
}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of a tcgen05 launch class, from the committed `ncu --set full`
# captures (profiler numbers, so they are constants here, never measured inside the timed region).  Key = the launch tag
# of ops._timed_call at R2 / batch 16.
NCU_TRAFFIC = {
    # round 2 capture of the dominant launch class (profiles/r02a_ncu_fused.txt): the gamma|beta convolution with the SPADE+Style
    # modulation in its epilogue, training variant (also writes gamma and the 1-bit activation mask)
    "fwd+spade B16 640x384 Cin128 Cout256 T9": (3.296e9,
        "ncu --set full (profiles/r02a_ncu_fused.txt): tapconv_fwd_kernel<256,0,2,0> (training variant), B16 640x384 128->256 3x3 + "
        "SPADE+Style epilogue: dram read 1.270 GB + write 2.025 GB per launch vs 3.34 GB algorithmic (actv 1.007 + x 0.252 at half "
        "resolution + out 1.007 + gamma 1.007 + mask 0.063); tensor pipe 66.8 % active at 1.51 GHz (power-capped). The no-grad "
        "variant <256,0,1,0> of the same class (D step / inference) moves 2.27 GB algorithmic. Re-measured on the final binaries "
        "inside a whole step (profiles/r02f_step_metrics_summary.txt): 1.266 GB read + 2.027 GB written, tensor pipe 63.3 %"),
    "fwd B16 640x384 Cin128 Cout256 T9": (2.982e9,
        "ncu --set full (profiles/r02a_ncu_conv256.txt): tapconv_fwd_kernel<256,0,0,0>, B16 640x384 128->256 3x3: dram read 1.022 GB "
        "+ write 1.960 GB per launch vs 3.020 GB algorithmic (x 1.007 GB + y 2.013 GB); tensor pipe 76.3 % active at 1.45 GHz"),
    "dgrad B16 640x384 Cin256 Cout128 T9": (2.998e9,
        "ncu --set full (profiles/r02a_ncu_conv256.txt): tapconv_fwd_kernel<128,0,0,0> as data gradient, B16 640x384 256->128 3x3: "
        "dram read 2.019 GB + write 0.979 GB per launch vs 3.020 GB algorithmic; tensor pipe 58.7 % (since round 2d this class "
        "runs the swapped-operand kernel <128,0,3,0>: same traffic, tensor pipe 77.9 %, profiles/r02d_ncu_swapped256to128.txt)"),
    "wgrad B16 640x384 Cin128 Cout256 T9": (3.749e9,
        "ncu --set full (profiles/r02a_ncu_conv256.txt): tapconv_wgrad_kernel<256>: dram read 3.743 GB + write 0.006 GB per launch "
        "vs 3.020 GB algorithmic (x 1.007 GB + dy 2.013 GB; 1.24x: taps whose CTAs are not co-resident re-read through DRAM); "
        "tensor pipe 58.2 %"),
}
# SPADE+Style normalisation kernels, launch B16 HW245760 C128 with the nearest-2x index map (profiles/r02b_ncu_norm.txt)
NCU_TRAFFIC_NORM_FWD = (3.281e9, "ncu --set full (profiles/r02b_ncu_norm.txt): spade_fwd_kernel<1,1>, B16 640x384 C128 reading x at half "
                        "resolution: dram read 2.265 GB + write 1.016 GB vs 3.27 GB algorithmic (x 0.25 + gamma|beta 2.01 + out 1.01); "
                        "77.6 % of ncu's DRAM peak, 6.35 TB/s")
NCU_TRAFFIC_NORM_BWD = (6.867e9, "ncu --set full (profiles/r02b_ncu_norm.txt): spade_bwd_reduce_kernel<1,1> 2.328 GB read (0.631 ms) + "
                        "spade_bwd_apply_kernel<1,1> 2.328 GB read + 2.208 GB written (0.773 ms) for the same launch: both passes read "
                        "dout, gamma and the 1-bit mask at full and x at half resolution; the apply pass writes dgamma|dbeta and the "
                        "half-resolution dx (2x2 adjoint of the up-sampling folded in)")


def ncu_traffic_for(tag, res, batch):
    """(bytes or None, note or None) for the dominant launch class of the bench workload."""
    if res != "R2" or batch != 16:
        return None, None
    return NCU_TRAFFIC.get(tag, (None, None))


def make_opts(res, batch, workload="c2"):
    from oracle import seg2eye_oracle as O
    crop, ar = RES[res]
    extra = dict(label_nc=35, netG="spade") if workload == "c5" else {}
    oopt = O.make_opt(crop_size=crop, aspect_ratio=ar, lambda_l1=10.0, **extra)
    d = vars(oopt).copy()
    d.update(gpu_ids=[0], init_type="xavier", init_variance=0.02, netD_subarch="n_layer", continue_train=False,
             which_epoch="latest", checkpoints_dir="/tmp/s2e_bench", name="bench", no_vgg_loss=True, lambda_openeds=0.0,
             lambda_style_w=0.0, lambda_style_feat=0.0, lambda_gram=0.0, netD="multiscale", batchSize=batch)
    d.setdefault("netG", "spadestyle")
    return oopt, SimpleNamespace(**d)


def workload_config(res, batch, world, workload="c2"):
    return {"workload": "%s, %s = %dx%d, per-GPU batch %d, ngf=ndf=64" % (
                WORKLOADS[workload], res, round(RES[res][0] / RES[res][1]), RES[res][0], batch),
            "baseline_config": {"c2": "BASELINE.json configs[1] (N = 1) / configs[2] (N > 1)", "c4": "BASELINE.json configs[3]",
                                "c5": "BASELINE.json configs[4]"}[workload],
            "global_batch": batch * world, "parallelism": "dp%d" % world,
            "l2_policy": "inputs+activations per step (>1 GB) exceed the 126 MB L2"}


DUMP_SAMPLE = 1 << 22   # an output with more elements is dumped as a fixed sample of this many (16 MB in float32)


def dump_outputs(out_dir, arrays):
    """<out_dir>/<name>.npy in float32 for each array; a larger one than DUMP_SAMPLE elements is replaced by the same
    seeded sample of its flattened elements (in index order) on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > DUMP_SAMPLE:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name.replace("/", "_") + ".npy"), a.numpy())


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in o.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference(res, steps, warmup, batch=1, keep_first=False, workload="c2"):
    """Oracle port of the reference step on the host cores; each step = one G step + one D step on `batch` images.
    keep_first: also return the losses / generated image of the FIRST iteration (from the initial weights) -- the
    reference side of the in-bench parity check."""
    from oracle import seg2eye_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    oopt, _ = make_opts(res, batch, workload)
    sd = parity_state(oopt)
    tr = O.OracleTrainer(sd["G"], sd["D"], sd["E"], oopt)
    b = O.synth_batch(oopt, batch, 1234)
    times, first = [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        tr.run_generator_one_step(b)
        tr.run_discriminator_one_step(b)
        dt = time.perf_counter() - t0
        if i == 0 and keep_first:
            first = ({k: float(v.reshape(-1)[0]) for k, v in {**tr.g_losses, **tr.d_losses}.items()}, tr.generated.detach().clone())
        if i >= warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    return dict(value=batch / (ms / 1e3), ms_per_step=ms, cores=torch.get_num_threads(), first=first,
                sample="%d G+D iteration(s) of batch %d at %s after %d warm-up" % (steps, batch, res, warmup))


def parity_state(oopt):
    """Reference-initialised weights (base_network.py:28-59) from portable seeds: the SAME state for the CPU arm and
    for the in-bench parity run of the CUDA path."""
    from oracle import seg2eye_oracle as O
    return dict(G=O.init_state(O.generator_shapes(oopt), 1), D=O.init_state(O.discriminator_shapes(oopt), 2),
                E=O.init_state(O.encoder_shapes(oopt), 3) if getattr(oopt, "netG", "spadestyle") != "spade" else {})


def parity_ours(res, first, batch=1, workload="c2"):
    """One G step + one D step of the CUDA path at the BENCH size (ngf = ndf = 64, `res`), batch `batch`, from the same
    weights and inputs as the oracle's first iteration; returns the comparison that goes into the JSON line.
    Tolerances: BASELINE.md section 5 / north_star (losses 2e-2 relative, GAN term with a 2e-2 absolute floor because it is
    a mean of signed logits that nearly cancels; image: chained bf16 bound, DESIGN.md section 2)."""
    import contextlib, io
    from oracle import seg2eye_oracle as O
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer
    oopt, opt = make_opts(res, batch, workload)
    opt.gpu_ids = [torch.cuda.current_device()]
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    m = tr.pix2pix_model
    sd = parity_state(oopt)
    for net, k in ((m.netG, "G"), (m.netD, "D"), (m.netE, "E")):
        if net is not None:
            net.load_state_dict({a: b.clone() for a, b in sd[k].items()})
            net.cuda()
    data = {k: v.clone() for k, v in O.synth_batch(oopt, batch, 1234).items()}
    if m.netE is None:
        data.pop("style_image")
    tr.run_generator_one_step(data)
    tr.run_discriminator_one_step(data)
    torch.cuda.synchronize()
    ours = {k: float(v.reshape(-1)[0]) for k, v in tr.get_latest_losses().items()}
    ref_losses, ref_img = first
    img = tr.generated.detach().float().cpu()
    img_err = float((img.double() - ref_img.double()).norm() / ref_img.double().norm())
    rows, ok = {}, True
    for k, r in ref_losses.items():
        tol = 2e-2 * abs(r) + (2e-2 if k == "GAN" else 0.0)
        rows[k] = {"ours": ours[k], "reference": r, "abs_err": abs(ours[k] - r), "tol": tol}
        ok = ok and abs(ours[k] - r) <= tol
    return {"config": "%s %s, batch %d, ngf=ndf=64, reference-initialised weights, first G+D iteration" % (workload, res, batch),
            "image_rel_l2_err": img_err, "image_tol": 2e-2, "losses": rows, "losses_tol": "2e-2 relative (+2e-2 absolute for GAN)",
            "pass": bool(ok and img_err <= 2e-2)}


# ------------------------------------------------------------------------------------------------ library arm (stock torch on the GPU)
def library_reference(res, steps, warmup, batch, precision, workload="c2"):
    """The SAME restatement of the reference step, executed by stock PyTorch on the B200 (cuDNN / cuBLAS / ATen): the
    "library baseline" of SURVEY 8(d) / BASELINE.md 6.5 -- what `--gpu_ids 0` of the reference costs on this GPU.
    precision: 'tf32' (fp32 storage, TF32 tensor cores -- torch's default for cuDNN convolutions) or 'bf16'
    (torch.autocast + channels_last).  Tries `batch` first and halves it on out-of-memory."""
    from oracle import seg2eye_oracle as O
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    cl = precision == "bf16"

    def to_dev(sd):
        out = {}
        for k, v in sd.items():
            t = v.to(dev)
            if cl and t.dim() == 4:
                t = t.contiguous(memory_format=torch.channels_last)
            out[k] = t
        return out

    b = batch
    while b >= 1:
        try:
            oopt, _ = make_opts(res, b, workload)
            sd = {k: to_dev(v) for k, v in parity_state(oopt).items()}
            tr = O.OracleTrainer(sd["G"], sd["D"], sd["E"], oopt)
            data = {k: v.to(dev) for k, v in O.synth_batch(oopt, b, 1234).items()}
            ctx = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if cl else (lambda: __import__("contextlib").nullcontext())

            def step():
                with ctx():
                    tr.run_generator_one_step(data)
                    tr.run_discriminator_one_step(data)
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            return dict(value=b / (ms / 1e3), ms_per_step=ms, batch=b, precision=precision,
                        peak_mem_gb=round(torch.cuda.max_memory_allocated() / 2**30, 1),
                        losses={k: float(v.reshape(-1)[0]) for k, v in {**tr.g_losses, **tr.d_losses}.items()})
        except torch.cuda.OutOfMemoryError:
            tr = sd = data = None
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            b //= 2
    raise RuntimeError("library baseline: batch 1 does not fit")


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch.distributed as dist
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import _lib as L, ops, parallel
    from seg2eye_b200.trainers.pix2pix_trainer import Pix2PixTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    oopt, opt = make_opts(args.res, args.batch, args.workload)
    opt.gpu_ids = [local]
    import contextlib, io
    torch.manual_seed(1234 + rank)      # replicas are made identical by the trainer itself (broadcast from rank 0)
    with contextlib.redirect_stdout(io.StringIO()):
        tr = Pix2PixTrainer(opt)
    m = tr.pix2pix_model
    nets = [net for net in (m.netG, m.netD, m.netE) if net is not None]
    seeded = [{k: v.clone() for k, v in net.state_dict().items()} for net in nets] if args.dump_outputs else None
    host = O.synth_batch(oopt, args.batch, 1234 + rank)
    if m.netE is None:
        host.pop("style_image")
    host = {k: v.pin_memory() for k, v in host.items()}
    dev = {k: v.cuda(non_blocking=True) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def step(data):
        d = dict(data)
        tr.run_generator_one_step(d)
        tr.run_discriminator_one_step(d)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(dev)
    barrier()

    # ---- per-kernel CUDA-event timing (eager pass; events cannot be attached to graph replays)
    ops.profile_begin()
    n0 = L.launches
    for _ in range(2):
        step(dev)
    launches_per_step = (L.launches - n0) // 2
    prof = ops.profile_end()
    barrier()
    if args.ncu_step:   # one eager step delimited by cudaProfilerStart/Stop (ncu --profile-from-start off)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step(dev)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    ms_eager = None
    if args.mode == "graph":
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(2):
            step(dev)
        t1.record(); torch.cuda.synchronize()
        ms_eager = t0.elapsed_time(t1) / 2
        tr.enable_cuda_graphs(dev, warmup=1)
        for _ in range(args.warmup):
            step(dev)
        barrier()

    # ---- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(dev)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = launches_per_step * args.steps
    # ---- timed region 2: end to end through the trainer API with host buffers
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d2h = 0
    f0.record()
    for _ in range(args.steps):
        step(host)
        vals = torch.stack([v.reshape(-1)[0] for v in tr.get_latest_losses().values()]).cpu()
        d2h = vals.numel() * 4
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    sampler.stop_flag = True
    sampler.join(2)
    if args.dump_outputs:
        # The weight-gradient and loss reductions add with float atomics, so a step is reproducible to rounding only, and
        # Adam(beta1 = 0) steps from the small initial weights amplify that: two seeded runs differ by 4e-3 in the image
        # after two steps and are unrelated after five (tools/trajectory_repro.py, profiles/r03_trajectory_repro.txt).  The
        # dumped step is therefore one more step of the timed path from the seeded weights and fresh optimizers, loaded the
        # way a checkpoint is (the graphs re-pack the bf16 weights themselves before the replay).
        for net, sd in zip(nets, seeded):
            net.load_state_dict(sd)
        tr.reset_optimizers()
        step(dev)
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, {"generated": tr.get_latest_generated(),
                                             **{"loss_" + k: v for k, v in tr.get_latest_losses().items()}})

    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    imgs = args.steps * args.batch * world
    peaks = load_peaks()
    out = None
    if rank == 0:
        conv_ms, conv_tf, conv_n = prof["tc_ms"], prof["tc_flop"] / 1e12, prof["tc_n"]
        achieved = conv_tf / (conv_ms / 1e3) if conv_ms > 0 else 0.0
        norm_gbs = prof["norm_bytes"] / 1e9 / (prof["norm_ms"] / 1e3) if prof["norm_ms"] > 0 else 0.0
        # the single launch class that takes the most time: the gamma|beta forward convolution at full resolution
        dom_tag, dom = max(((t, v) for (k, t), v in prof["by_tag"].items() if k == "tc"), key=lambda kv: kv[1][1])
        dominant = {"launch": dom_tag, "launches_per_step": dom[0] // 2, "ms_per_launch": dom[1] / dom[0],
                    "tflops": dom[2] / 1e12 / (dom[1] / 1e3)}
        traffic, traffic_note = ncu_traffic_for(dom_tag, args.res, args.batch)
        traffic_launch = dom_tag
        if traffic is None:   # the dominant class has no ncu capture yet: report the largest class that has one, and say so
            captured = [(v[1], t) for (k, t), v in prof["by_tag"].items() if k == "tc" and ncu_traffic_for(t, args.res, args.batch)[0]]
            if captured:
                traffic_launch = max(captured)[1]
                note_dom = traffic_note
                traffic, traffic_note = ncu_traffic_for(traffic_launch, args.res, args.batch)
                traffic_note = "launch class '%s' (largest class with an ncu capture): %s || dominant class '%s': %s" % (
                    traffic_launch, traffic_note, dom_tag, note_dom)
        out = {
            "metric": "G+D train images/sec", "value": imgs / (ms / 1e3), "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args.res, args.batch, world, args.workload),
            "e2e": {"value": imgs / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches,
            "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1),
            "execution": (("2 CUDA graphs per iteration (G step, D step)" if world == 1 else
                           "4 CUDA graphs per iteration ([fwd+bwd], [Adam] for G and D) with the NCCL gradient all-reduce between them")
                          + "; eager ms_per_step %.1f" % ms_eager) if ms_eager else "eager",
            "clocks": sampler.summary(),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": achieved / peaks["tf_sustained"], "traffic": traffic, "traffic_launch": traffic_launch, "traffic_note": traffic_note,
                         "dominant": dominant,
                         "kernel": "tapconv_{fwd,wgrad}_kernel (tcgen05 implicit GEMM; %d launches/step, %.1f ms of the %.1f ms step; "
                                   "CUDA events around each launch in a 2-step eager pass)" % (
                             conv_n // 2, conv_ms / 2, ms / args.steps),
                         "peak_source": peaks["source"] + " (sustained bf16 cuBLAS; burst %.0f)" % peaks["tf"]},
            "roofline_norm": {"bound": "hbm", "achieved": norm_gbs, "peak": peaks["hbm"], "unit": "GB/s",
                              "frac": norm_gbs / peaks["hbm"], "kernel": "spade_fwd_kernel (8 B/element: x, gamma, beta in, out; the SPADE blocks with C <= 128 run inside the gamma|beta "
                                        "convolution's epilogue instead and are counted under `roofline`)",
                              "launches": prof["norm_n"],
                              "traffic": NCU_TRAFFIC_NORM_FWD[0], "traffic_note": NCU_TRAFFIC_NORM_FWD[1]},
        }
        if prof.get("normb_ms", 0) > 0:
            nb = prof["normb_bytes"] / 1e9 / (prof["normb_ms"] / 1e3)
            out["roofline_norm_bwd"] = {"bound": "hbm", "achieved": nb, "peak": peaks["hbm"], "unit": "GB/s", "frac": nb / peaks["hbm"],
                                        "kernel": "spade_style_bwd (reduce + fold + apply; 12 B/element algorithmic: dout, x, gamma in; "
                                                  "dx, dgamma, dbeta out)", "launches": prof["normb_n"],
                                        "traffic": NCU_TRAFFIC_NORM_BWD[0], "traffic_note": NCU_TRAFFIC_NORM_BWD[1]}
        if args.workload == "c2" and args.res in STEP_TFLOP:
            out["step_tflops_equiv"] = imgs * STEP_TFLOP[args.res] / (ms / 1e3)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------ config 4: inference sweep
def run_c4(args):
    """BASELINE config 4 (SURVEY 8(d) C4): mode='encode_only' on two style sets -> linear interpolation of w in `batch`
    steps -> mode='inference' with latent_style (batch, 16) and the label repeated -> device tail (640x400 integers, what
    util/tester.py:44-47 produces on the host).  One step = one sweep = `batch` generated images.  Single GPU (replicas
    only: independent sweeps)."""
    import contextlib, io
    from oracle import seg2eye_oracle as O
    from seg2eye_b200 import _lib as L, ops, postprocessor
    from seg2eye_b200.models.pix2pix_model import Pix2PixModel
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    nb = args.batch
    oopt, opt = make_opts(args.res, nb, "c2")
    opt.gpu_ids = [local]
    torch.manual_seed(1234)
    with contextlib.redirect_stdout(io.StringIO()):
        m = Pix2PixModel(opt)
    m.eval()      # test.py: model.eval() -- BatchNorm running statistics, no spectral-norm iteration
    b2 = O.synth_batch(oopt, 2, 1234)
    host = {"label": b2["label"][0:1].repeat(nb, 1, 1, 1).contiguous().pin_memory(), "style_image": b2["style_image"].pin_memory()}
    dev = {k: v.cuda() for k, v in host.items()}
    alphas = torch.linspace(0, 1, nb, device="cuda").view(-1, 1)
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def sweep(data, tail):
        with torch.no_grad():
            w = m({"label": data["label"][:2], "style_image": data["style_image"]}, mode="encode_only")
            wi = (1 - alphas) * w[0:1] + alphas * w[1:2]
            fake = m({"label": data["label"], "style_image": data["style_image"], "latent_style": wi}, mode="inference")
            return postprocessor.ImageProcessor.to_255resized_imagebatch(fake) if tail else fake

    for _ in range(args.warmup):
        sweep(dev, True)
    torch.cuda.synchronize()
    ops.profile_begin()
    n0 = L.launches
    sweep(dev, True)
    launches = L.launches - n0
    prof = ops.profile_end()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        sweep(dev, True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out_host = torch.empty(nb, 1, 640, 400, dtype=torch.int32).pin_memory()
    f0.record()
    for _ in range(args.steps):
        d = {k: v.cuda(non_blocking=True) for k, v in host.items()}
        out_host.copy_(sweep(d, True), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    f1.record()
    torch.cuda.synchronize()
    ms_e2e = f0.elapsed_time(f1)
    sampler.stop_flag = True
    sampler.join(2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": out_host})
    peaks = load_peaks()
    conv_ms, conv_tf = prof["tc_ms"], prof["tc_flop"] / 1e12
    achieved = conv_tf / (conv_ms / 1e3) if conv_ms > 0 else 0.0
    dom_tag, dom = max(((t, v) for (k, t), v in prof["by_tag"].items() if k == "tc"), key=lambda kv: kv[1][1])
    imgs = args.steps * nb
    out = {"metric": "inference images/sec (style-interpolation sweep)", "value": imgs / (ms / 1e3), "unit": "images/s", "n_gpus": 1,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args.res, nb, 1, "c4"),
           "e2e": {"value": imgs / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": out_host.numel() * 4},
           "gpu_launches": launches * args.steps, "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1),
           "execution": "eager, no-grad (gamma|beta convolutions with the SPADE+Style modulation fused into their epilogues)",
           "clocks": sampler.summary(),
           "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": achieved / peaks["tf_sustained"], "traffic": None,
                        "dominant": {"launch": dom_tag, "launches_per_step": dom[0], "ms_per_launch": dom[1] / dom[0],
                                     "tflops": dom[2] / 1e12 / (dom[1] / 1e3)},
                        "kernel": "tapconv_fwd_kernel (tcgen05; %d launches/sweep, %.1f ms of the %.1f ms sweep)" % (
                            prof["tc_n"], conv_ms, ms / args.steps),
                        "peak_source": peaks["source"] + " (sustained bf16 cuBLAS; burst %.0f)" % peaks["tf"]}}
    if not args.no_cpu_baseline:
        # oracle port on the host cores: encode two style sets + generator forward of a 4-image slice of the sweep
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sd = parity_state(oopt)
        t0 = time.perf_counter()
        with torch.no_grad():
            w = O.encode_w(sd["E"], b2["style_image"], oopt, training=False)
            wi = torch.stack([w[0] * (1 - a) + w[1] * a for a in (0.0, 0.33, 0.66, 1.0)])
            ref = O.generator_forward(sd["G"], O.one_hot(b2["label"][0:1].repeat(4, 1, 1, 1), 4), wi, oopt, training=False)
            O.to_255_resized(ref)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 4 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                               "sample": "encode 2 style sets + 4 of the %d interpolated images + host tail, once, at %s" % (nb, args.res)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference", "library"))
    ap.add_argument("--workload", default="c2", choices=tuple(WORKLOADS))
    ap.add_argument("--res", default=None, choices=tuple(RES))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--mode", default="graph", choices=("graph", "eager"))
    ap.add_argument("--ncu-step", action="store_true", help="bracket one eager step with cudaProfilerStart/Stop")
    ap.add_argument("--precision", default="bf16", choices=("bf16", "tf32"), help="--impl library only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of one step of the timed path, from the seeded "
                    "weights, to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    if args.res is None:
        args.res = {"c2": "R2", "c4": "R1", "c5": "S256"}[args.workload]
    if args.batch is None:
        args.batch = {"c2": 16, "c4": 64, "c5": 16}[args.workload]

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = args.steps, args.warmup
        r = cpu_reference(args.res, steps, warmup, workload=args.workload)
        cb = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
              "sample": r["sample"] + " (oracle/seg2eye_oracle.py: fp32 PyTorch-CPU restatement of the reference; the reference "
                                      "itself is Python and its checkout does not exist on the GPU box)"}
        cfg = workload_config(args.res, args.batch, max(1, args.gpus), args.workload)
        cfg["sample_batch"] = 1    # the CPU arm times a bounded sample of the workload: batch 1 per step, images/s is per image
        print(json.dumps({
            "impl": "reference", "metric": "G+D train images/sec", "value": r["value"], "unit": "images/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": cfg, "cpu_baseline": cb,
            "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    if args.impl == "library":
        if rank != 0:
            return
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        r = library_reference(args.res, args.steps, args.warmup, args.batch, args.precision, args.workload)
        print(json.dumps({
            "impl": "library", "metric": "G+D train images/sec", "value": r["value"], "unit": "images/s", "n_gpus": 1,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args.res, r["batch"], 1, args.workload), "peak_mem_gb": r["peak_mem_gb"], "losses": r["losses"],
            "note": "stock PyTorch (cuDNN/cuBLAS/ATen) executing the reference step on the same B200: %s" % (
                "fp32 storage, TF32 convolutions" if args.precision == "tf32" else "torch.autocast(bf16) + channels_last")}))
        return

    assert args.warmup >= 3, "timing rule: at least 3 warm-up steps"
    if args.workload == "c4":
        if rank == 0:
            print(json.dumps(run_c4(args)))
        return
    out = run_ours(args)
    if rank == 0:
        if int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline:
            # rank 0, N = 1 only: the oracle port on the host cores; its first iteration doubles as the parity reference
            r = cpu_reference(args.res, 2, 1, keep_first=True, workload=args.workload)
            out["cpu_baseline"] = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                                   "sample": r["sample"]}
            try:
                out["parity"] = parity_ours(args.res, r["first"], workload=args.workload)
            except Exception as e:   # the bench line must still be printed; a failed parity run is reported as such
                out["parity"] = {"pass": False, "error": repr(e)[:300]}
        if int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_library_baseline:
            # the library baselines run in their own processes so that their allocator / cuDNN workspaces never share
            # the measured process
            lib = {}
            for prec in ("bf16", "tf32"):
                try:
                    o = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "library", "--precision", prec,
                                        "--workload", args.workload, "--res", args.res, "--batch", str(args.batch), "--steps", "3", "--warmup", "2"],
                                       capture_output=True, text=True, timeout=600)
                    line = [l for l in o.stdout.splitlines() if l.startswith("{")][-1]
                    d = json.loads(line)
                    lib[prec] = {"value": d["value"], "unit": "images/s", "batch": d["config"]["global_batch"],
                                 "ms_per_step": d["ms_per_step"], "peak_mem_gb": d["peak_mem_gb"],
                                 "ratio_ours_over_library": out["value"] / d["value"]}
                except Exception as e:
                    lib[prec] = {"unavailable": repr(e)[:200]}
            out["library_baseline"] = lib
        print(json.dumps(out))


if __name__ == "__main__":
    main()
