#!/usr/bin/env python
"""bench.py -- volumes/sec of the 3D U-Net hot path on B200.

  python bench.py --gpus N --steps K --warmup W [--config C2|C3|C5]     B200 arm (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K ...               the reference's CPU implementation of the path
  python bench.py ... --dump-outputs DIR                                 also write what the last timed step computed, DIR/<name>.npy

Workloads (BASELINE.json `configs`): C2 (default, configs[1], the one `metric` is quoted on): 4-channel 128^3 volumes,
UNet3D base_width=32, bf16 tensor-core operands / fp32 accumulate, batch 2 per GPU, one step = forward, sigmoid-Dice,
backward, [gradient all-reduce,] fused Adam.  C3 (configs[2]): the same at 160x192x128.  C5 (configs[4]): 1-channel 256^3
5-level base_width=48 tiled inference (SlidingWindowInferer 128^3, overlap 0.25 = 27 tiles).  Synthetic data, random-init weights.

Prints ONE JSON line on rank 0.  `value`: inputs resident in HBM, CUDA-event timed, max over ranks; the step is replayed
as a CUDA graph (train.GraphedTrainStep).  `e2e`: the same work through the reference-facing API
(train.epoch_training(..., use_cuda_graph=True) / predict.volumetric_predictions) from pinned HOST buffers, H2D (and the
result's D2H) inside the timed region.  `roofline`: the halo-resident implicit-GEMM convolution kernel k_conv_halo (the
dominant kernel), algorithmic FLOPs / CUDA-event time summed over its launches against the measured bf16 peak.
`cpu_baseline`: the oracle port of the reference model (torch CPU ops) on a bounded sample.  `cudnn_baseline`: the same
op graph through torch/cuDNN under bf16 autocast on this GPU, timed in the same run (the bar SURVEY.md 8d names).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "volumes/s"

# BASELINE.json configs: C2 = configs[1] (the config `metric` is quoted on; default), C3 = configs[2], C5 = configs[4].
CONFIGS = {
    "C2": dict(kind="train", model=dict(n_features=4, n_outputs=3, base_width=32), volume=(128, 128, 128), batch=2,
               metric="volumes/sec fwd+bwd 4ch 128^3 UNet",
               workload="C2: 4ch 128^3 UNet3D base_width=32, fwd + sigmoid-Dice + bwd + fused Adam, batch 2 per GPU"),
    "C3": dict(kind="train", model=dict(n_features=4, n_outputs=3, base_width=32), volume=(160, 192, 128), batch=2,
               metric="volumes/sec fwd+bwd 4ch 160x192x128 UNet",
               workload="C3: 4ch 160x192x128 (BraTS full patch) UNet3D base_width=32, fwd + sigmoid-Dice + bwd + fused Adam, "
                        "batch 2 per GPU"),
    "C5": dict(kind="infer", model=dict(n_features=1, n_outputs=1, base_width=48, encoder_blocks=[1, 2, 2, 4, 4]),
               volume=(256, 256, 256), batch=1, roi=(128, 128, 128), overlap=0.25, sw_batch=3,
               metric="volumes/sec tiled inference 1ch 256^3 5-level UNet width 48",
               workload="C5: 1ch 256^3 5-level UNet3D base_width=48 inference, SlidingWindowInferer roi 128^3 overlap 0.25 "
                        "(27 tiles, 3 per forward) through predict.volumetric_predictions"),
}

# mean DRAM bytes per k_conv_halo launch in one C2 training step (ncu launch list under profiles/); refresh with
# tools/gpu_trip_prof.sh + tools/summarize_ncu.py when the kernel or the dispatch changes
NCU_TRAFFIC = {"bytes_per_launch": 339.6e6, "source": "profiles/r02_launches.txt (ncu dram__bytes_read.sum + dram__bytes_write.sum, "
                                                      "mean over the kernel's launches of one C2 step)"}


# --dump-outputs keeps at most this many elements of one array (16 MiB in float32), so that a dump stays under 64 MB
DUMP_SAMPLE = 1 << 22


def dump_outputs(path, arrays):
    """Writes each tensor as float32 ``path/<name>.npy``.  A tensor of more than DUMP_SAMPLE elements is replaced by its
    flattened elements at DUMP_SAMPLE fixed positions (the first entries of a seed-0 permutation, ascending), the same
    positions in every run of the same workload, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"tflops": float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1590.0))), "hbm_gbs": float(p.get("hbm_gbs", 6650.0)),
                "source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"}
    return {"tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md): 1.59 PFLOP/s, 6.65 TB/s"}


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [c.strip() for c in line.split(",")]
                if len(f) >= 9:
                    rows.append(f)
            os.unlink(self.path)
        except Exception:
            pass
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out.update(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=float(rows[0][2]) if rows[0][2].replace(".", "").isdigit() else None,
                   reasons=sorted(reasons), samples=len(rows), power_w_max=max(float(r[3]) for r in rows if r[3].replace(".", "").isdigit()))
        return out


def synth_batch(cfg, batch, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((batch, cfg["model"]["n_features"]) + cfg["volume"], generator=g, dtype=torch.float32)
    t = (torch.rand((batch, cfg["model"]["n_outputs"]) + cfg["volume"], generator=torch.Generator().manual_seed(seed + 1)) > 0.7).to(torch.uint8)
    return x, t


# ------------------------------------------------------------------------------------------------ reference (CPU) arm
def cpu_reference_throughput(cfg, steps, warmup, budget_s=150.0, batch=1):
    """The oracle port (torch CPU ops == the reference's arithmetic library; the live reference module when it is
    mounted) on the host cores.  Each step is a bounded sample: a crop of one volume (training configs: fwd + Dice + bwd;
    C5: the forward of a crop of one 128^3 tile, scaled to the 27 tiles of a volume) sized so that (steps + warmup) steps
    fit `budget_s`.  Thread count: swept over {16, 32, 64, all cores} ON A 64^3 CROP of the timed workload (one warm-up +
    one timed step each), the fastest is used and reported as `cores`."""
    from oracle import UNetConfig, make_state_dict, unet3d_forward, dice_loss
    from oracle.ref_loader import reference_available
    mkw = cfg["model"]
    ocfg = UNetConfig(**mkw)
    train = cfg["kind"] == "train"
    kind = "port"
    model = None
    if reference_available():
        try:
            from oracle.ref_loader import reference_unet3d
            model = reference_unet3d(**mkw)
            model.train(train)
            model.encoder.layers[0].dropout.p = 0.0
            kind = "reference"
        except Exception:
            model = None
    sd = {k: v.requires_grad_(train) for k, v in make_state_dict(ocfg, seed=0).items()}

    def step(shape):
        g = torch.Generator().manual_seed(1)
        x = torch.randn((batch, ocfg.n_features) + shape, generator=g)
        t = (torch.rand((batch, ocfg.n_outputs) + shape, generator=g) > 0.7).to(torch.uint8)
        t0 = time.perf_counter()
        if not train:
            with torch.no_grad():
                model(x) if model is not None else unet3d_forward(sd, x, ocfg)
            return time.perf_counter() - t0
        if model is not None:
            model.zero_grad(set_to_none=True)
            loss = dice_loss(model(x), t)
        else:
            for p in sd.values():
                p.grad = None
            loss = dice_loss(unet3d_forward(sd, x, ocfg), t)
        loss.backward()
        return time.perf_counter() - t0

    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    probe = (64, 64, 64)
    sweep = []
    for nt in sorted({min(ncpu, 16), min(ncpu, 32), min(ncpu, 64), ncpu}):
        torch.set_num_threads(nt)
        step(probe)
        sweep.append((step(probe), nt))
    sweep.sort()
    t64, nthreads = sweep[0]
    torch.set_num_threads(nthreads)
    unit = cfg["volume"] if train else cfg["roi"]        # the volume (or tile) a crop is a fraction of
    full = unit[0] * unit[1] * unit[2]
    crops = [unit, (unit[0], unit[1], unit[2] // 2), (unit[0], unit[1] // 2, unit[2] // 2), (64, 64, 64), (64, 64, 32), (64, 32, 32), (32, 32, 32)]
    chosen = crops[-1]
    for c in crops:
        est = t64 * (c[0] * c[1] * c[2]) / 64 ** 3
        if est * (steps + warmup) <= budget_s:
            chosen = c
            break
    frac = chosen[0] * chosen[1] * chosen[2] / full
    # the two fastest thread counts of the 64^3 probe are re-timed AT THE REPORTED SIZE (one step each) when the budget allows
    resweep = ""
    est = t64 * (chosen[0] * chosen[1] * chosen[2]) / 64 ** 3
    if len(sweep) > 1 and est * (steps + warmup + 2) <= 1.5 * budget_s:
        at_size = []
        for _, nt in sweep[:2]:
            torch.set_num_threads(nt)
            at_size.append((step(chosen), nt))
        at_size.sort()
        nthreads = at_size[0][1]
        torch.set_num_threads(nthreads)
        resweep = "; the two fastest re-timed at the reported crop: " + ", ".join("%d threads %.1f s" % (nt, tt) for tt, nt in at_size)
    for _ in range(warmup):
        step(chosen)
    times = [step(chosen) for _ in range(steps)]
    total = sum(times)
    units_per_volume = 1 if train else 27
    vps = batch * frac * steps / total / units_per_volume
    what = "fwd+Dice+bwd" if train else "forward (no_grad)"
    of = "a %dx%dx%d volume" % unit if train else "one %dx%dx%d tile; a volume = 27 tiles" % unit
    return {"value": vps, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%d step(s) of %s on a %dx%dx%d crop (%.4g of %s), batch %d, fp32, %.1f s/step; threads = fastest of "
                      "{16,32,64,all} on a 64^3 crop%s" % (steps, what, chosen[0], chosen[1], chosen[2], frac, of, batch, total / steps, resweep)}, total / steps * 1e3


def run_reference_arm(args):
    rank, world, _ = env_rank()
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    cb, ms = cpu_reference_throughput(cfg, args.steps, args.warmup)
    line = {"impl": "reference", "metric": cfg["metric"], "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"].split(",")[0] + " on host CPU cores (bounded sample per step)", "sample": cb["sample"]},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ cuDNN bar (same GPU)
def cudnn_baseline(cfg, dev, steps=3):
    """The reference model's op graph (the oracle's functional restatement: the same torch ops the reference nn.Module
    issues) through torch/cuDNN under bf16 autocast on this GPU: the 'reference cuDNN 1-GPU volumes/sec' bar."""
    from oracle import UNetConfig, make_state_dict, unet3d_forward, dice_loss
    ocfg = UNetConfig(**cfg["model"])
    train = cfg["kind"] == "train"
    torch.backends.cudnn.benchmark = True
    try:
        sd = {k: v.to(dev).requires_grad_(train) for k, v in make_state_dict(ocfg, seed=0).items()}
        if train:
            x, t = synth_batch(cfg, cfg["batch"], seed=7)
            x, t = x.to(dev), t.to(dev)

            def step():
                for p in sd.values():
                    p.grad = None
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    out = unet3d_forward(sd, x, ocfg)
                loss = dice_loss(out.float(), t)
                loss.backward()
            vols = cfg["batch"]
        else:
            roi = cfg["roi"]
            tiles = torch.randn((cfg["sw_batch"], ocfg.n_features) + roi, device=dev)

            def step():          # 27 tiles of one volume, sw_batch per forward (tiling itself not included)
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                    for _ in range(27 // cfg["sw_batch"]):
                        unet3d_forward(sd, tiles, ocfg)
            vols = 1
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out = {"value": vols / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "kind": "torch %s + cuDNN %s, bf16 autocast, cudnn.benchmark=True, "
               "the oracle's functional graph of the reference model" % (torch.__version__, torch.backends.cudnn.version()), "steps": steps}
    except Exception as e:  # noqa: BLE001  (a baseline that cannot run is reported, not fatal)
        out = {"value": None, "error": repr(e)[:300]}
    torch.backends.cudnn.benchmark = False
    del sd
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ B200 arm
class _Meta(torch.Tensor):
    """Minimal MetaTensor stand-in: volumetric_predictions requires ``.meta['filename_or_obj']`` (volumetric.py:11-51)."""
    meta = None


def run_b200_arm(args):
    import torch.distributed as dist
    pkg = importlib.import_module("3dunetcnn_b200")
    rank, world, local = env_rank()
    cfg = CONFIGS[args.config]
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        pkg.parallel.init_process_group_from_env("nccl")
    if args.gpus != world and rank == 0:
        print("bench.py: --gpus %d but WORLD_SIZE=%d (launch N>1 with torch.distributed.run); using WORLD_SIZE" % (args.gpus, world), file=sys.stderr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Milliseconds of ``steps`` calls of ``fn`` (max over ranks) and what the last call returned."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item()), last

    torch.manual_seed(0)
    model = pkg.UNet3D(precision=args.precision, **cfg["model"]).to(dev)
    batch = cfg["batch"]
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local)
    extra = {}
    overlapped = False

    if cfg["kind"] == "train":
        crit = pkg.DiceLoss(sigmoid=True, include_background=True)
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)
        sync = pkg.parallel.GradAllReduce(model.parameters(), model=model)
        sync.broadcast_parameters(0)
        model.train()
        xh, th = synth_batch(cfg, batch, seed=100 + rank)
        x, t = xh.to(dev), th.to(dev)
        use_graph = not args.no_graph
        if use_graph:
            try:
                gstep = pkg.train.GraphedTrainStep(model, crit, opt, x.shape, t.shape, grad_sync=sync)
                gstep(x, t)                               # captures; a failure here falls back to eager launches below
                torch.cuda.synchronize()
            except Exception as e:  # noqa: BLE001  (both step drivers are product paths; say which one was measured)
                print("bench.py: CUDA-graph capture failed (%r); measuring the eager step loop instead" % (e,), file=sys.stderr)
                use_graph = False
                model._overwrite_grads = False
                model.__dict__.pop("_graphed_steps", None)
        if use_graph:
            overlapped = gstep.graph_tail is not None and world > 1

            def step_resident():
                return gstep(x, t)
        else:
            model.use_flat_gradients(True)

            def step_resident():
                opt.zero_grad(set_to_none=True)
                loss = crit(model(x), t)
                loss.backward()
                sync()
                opt.step()
                return loss

        for _ in range(warmup):
            step_resident()
        if rank == 0:
            sampler.start()
        ms_total, loss = timed(step_resident, args.steps)
        if args.dump_outputs and rank == 0:
            # what the step hands its caller: the loss, the gradients (flat, in state-dict order) and the updated parameters
            params = model.ordered_parameters()
            dump_outputs(args.dump_outputs, {"loss": loss, "gradients": torch.cat([p.grad.reshape(-1) for p in params]),
                                             "parameters": torch.cat([p.detach().reshape(-1) for p in params])})
        plan = model._plan_for(x)
        launches_per_step = model.launches_last_forward + model.launches_last_backward + 3   # + Dice sums/finalize/bwd

        # ---- e2e: the reference-facing step loop (training_utils.epoch_training) over K pinned host batches: H2D of every
        # batch and the read-back of every step's loss are inside the timed region
        loader = [{"image": xh.clone().pin_memory(), "label": th.clone().pin_memory()} for _ in range(2)]
        loader = [loader[i % 2] for i in range(args.steps)]

        def epoch():
            return pkg.train.epoch_training(loader, model, crit, opt, epoch=0, n_gpus=1, print_frequency=0, grad_sync=sync,
                                            use_cuda_graph=use_graph)
        pkg.train.epoch_training(loader[:3], model, crit, opt, epoch=0, n_gpus=1, print_frequency=0, grad_sync=sync,
                                 use_cuda_graph=use_graph)
        ms_e2e, _ = timed(epoch, 1)
        clocks = sampler.stop() if rank == 0 else None
        h2d = int(xh.numel() * 4 + th.numel())
        d2h = 4
        api = ("train.epoch_training(loader, model, criterion, optimizer, ..., use_cuda_graph=%s): pinned host batches, H2D one batch ahead "
               "on a copy stream, loss read back every step (one step behind the queue)" % use_graph)

        def profiled_step():
            opt.zero_grad(set_to_none=True)
            loss = crit(model(x), t)
            loss.backward()
        model._overwrite_grads = False
        vols_per_step = batch
    else:
        # ---- C5: tiled inference of one volume per step
        use_graph = False
        model.eval()
        inf = pkg.SlidingWindowInferer(roi_size=cfg["roi"], sw_batch_size=cfg["sw_batch"], overlap=cfg["overlap"])
        xh = torch.randn((batch, cfg["model"]["n_features"]) + cfg["volume"], generator=torch.Generator().manual_seed(100 + rank))
        x = xh.to(dev)

        def step_resident():
            with torch.no_grad():
                return inf(x, model)
        for _ in range(warmup):
            step_resident()
        if rank == 0:
            sampler.start()
        ms_total, prediction = timed(step_resident, args.steps)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"prediction": prediction})
        tiles = torch.empty((cfg["sw_batch"], cfg["model"]["n_features"]) + cfg["roi"], device=dev)
        plan = model._plan_for(tiles, inference_only=True)
        n_fwd = 27 // cfg["sw_batch"]
        launches_per_step = n_fwd * (model.launches_last_forward + 2) + 1
        # ---- e2e: predict.volumetric_predictions (volumetric.py:131-177) on a pinned host volume; the prediction is copied
        # back into pinned host memory by the writer (the reference writes NIfTI there)
        xp = xh.clone().pin_memory().as_subclass(_Meta)
        xp.meta = {"filename_or_obj": ["synthetic_%d.nii.gz" % i for i in range(batch)]}
        host_out = torch.empty((cfg["model"]["n_outputs"],) + cfg["volume"], dtype=torch.float32).pin_memory()

        def writer(fn, pred, out_dir):
            host_out.copy_(pred, non_blocking=True)

        def e2e_step():
            pkg.volumetric_predictions(model, [{"image": xp}], None, activation="sigmoid", inferer=inf, writer=writer)
        e2e_step()
        ms_e2e, _ = timed(e2e_step, args.steps)
        clocks = sampler.stop() if rank == 0 else None
        h2d = int(xh.numel() * 4)
        d2h = int(host_out.numel() * 4)
        api = "predict.volumetric_predictions(model, loader, dir, activation='sigmoid', inferer=SlidingWindowInferer(...), writer): pinned host volume in, pinned host prediction out"

        def profiled_step():
            with torch.no_grad():
                inf(x, model)
        vols_per_step = batch
        extra["tiles_per_volume"] = 27

    # ---- per-kernel accounting (CUDA events around every launch of the plan), same K steps repeated eagerly
    macs = plan.algorithmic_macs()
    reps = n_fwd if cfg["kind"] == "infer" else 1
    plan.profile_begin(args.steps * (launches_per_step + 16))
    for _ in range(args.steps):
        profiled_step()
    torch.cuda.synchronize()
    prof = plan.profile_end()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    vols = vols_per_step * world * args.steps
    value = vols / (ms_total / 1e3)
    e2e_steps = args.steps
    e2e_value = vols_per_step * world * e2e_steps / (ms_e2e / 1e3)
    conv_ms = prof["conv_halo"]["ms"]
    conv_launches = prof["conv_halo"]["launches"]
    conv_flops = 2.0 * macs["conv_halo"] * args.steps * reps
    achieved = conv_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
    conv_keys = ("conv_halo", "conv_fwd", "conv_dgrad", "conv_wgrad")
    all_conv_ms = sum(prof[k]["ms"] for k in conv_keys)
    all_conv_flops = 2.0 * sum(macs[k] for k in conv_keys) * args.steps * reps
    kernels = {}
    for k, v in prof.items():
        if v["launches"]:
            kernels[k] = {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps}
            if macs.get(k):
                kernels[k]["tflops"] = 2.0 * macs[k] * args.steps * reps / (v["ms"] / 1e3) / 1e12
    step_flops = 2.0 * sum(macs.values()) * reps
    whole_frac = step_flops / (ms_total / args.steps / 1e3) / 1e12 / peaks["tflops"]
    line = {
        "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "bf16x3-split", "data": "synthetic",
        "config": {"workload": cfg["workload"], "global_batch": batch * world, "volume": list(cfg["volume"]), "parallelism": "dp%d" % world,
                   "l2": "no flush: each step streams several GB of activations through HBM (>> 126 MB L2); every tensor is re-read from HBM",
                   "step": ("CUDA-graph replay of forward+Dice+backward (train.GraphedTrainStep), eager fused Adam" if cfg["kind"] == "train" and use_graph
                            else "eager launches"),
                   "grad_sync": (("in-place NCCL all-reduce (AVG) of the flat gradient bucket in two slices: head/decoder/deepest-encoder gradients (~90 % of the "
                                 "parameters) on a side stream under the backward of the shallow encoder levels (second CUDA graph), the rest after it"
                                 if overlapped else "in-place NCCL all-reduce (AVG) of the flat gradient bucket after backward") if world > 1 else "none")
                   if cfg["kind"] == "train" else "n/a (replicas)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / e2e_steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": api},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "k_conv_halo (halo-resident implicit-GEMM conv: forward + data-gradient launches)",
                     "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                     "traffic": NCU_TRAFFIC["bytes_per_launch"] if args.config == "C2" else None, "traffic_source": NCU_TRAFFIC["source"],
                     "all_conv_kernels_tflops": all_conv_flops / (all_conv_ms / 1e3) / 1e12 if all_conv_ms > 0 else 0.0,
                     "launches_per_step": conv_launches / args.steps, "ms_per_step": conv_ms / args.steps,
                     "peak_source": peaks["source"],
                     "timing": "CUDA-event pair around every launch on the launching stream, K eager steps repeated after the timed region",
                     "whole_step_frac_of_peak": whole_frac},
        "kernels": kernels,
        "algorithmic_flop_per_volume": step_flops / vols_per_step,
    }
    line.update(extra)
    if cfg["kind"] == "infer":
        line["roofline"]["volumes_per_s_at_peak"] = peaks["tflops"] * 1e12 / (step_flops / vols_per_step)
    if world == 1 and not args.no_cpu_baseline:
        del model
        torch.cuda.empty_cache()
        line["cudnn_baseline"] = cudnn_baseline(cfg, dev)
        cb, _ = cpu_reference_throughput(cfg, steps=1, warmup=0, budget_s=30.0)
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "split"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the CUDA-graph replayed step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as float32 "
                    "DIR/<name>.npy (training: loss, gradients, parameters; inference: prediction), at most %d elements each "
                    "(a fixed sample of a larger array)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
