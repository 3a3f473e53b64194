#!/usr/bin/env python
"""bench.py -- GANgealing train images/sec at 256^2 (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus 1 --steps K --warmup W              # this repo's sm_100a path
  torchrun ... bench.py --gpus N --steps K --warmup W        # one rank per GPU, NCCL (the driver launches this)
  python bench.py --impl reference ...                       # the reference algorithm on the host CPU cores

A "step" is one full training iteration of BASELINE config 2 (LSUN-Cats-256 recipe: frozen StyleGAN2-256
generator forward x2, similarity+flow STN @128, perceptual loss, backward, Adam x2, EMA, loss reduce) on a
synthetic batch (seeded random weights, z ~ N(0,1); no datasets or checkpoints exist offline).
Rank 0 prints ONE JSON line; see README / DESIGN.md for the field definitions.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "gangealing_train_images_per_sec_256"
UNIT = "images/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("GG_BENCH_BATCH", "32")), help="per-GPU batch")
    ap.add_argument("--cpu-batch", type=int, default=2, help="batch of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of as a CUDA graph")
    ap.add_argument("--dtype", default=os.environ.get("GG_BENCH_DTYPE", "f32"), choices=["f32", "bf16"],
                    help="activation storage type: f32 = BASELINE config 2 (the headline), bf16 = config 3")
    ap.add_argument("--no-extra", action="store_true", help="skip the additional config-3 (bf16) measurement of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy; the run then uses cuDNN's deterministic "
                         "algorithms (config.cudnn in the result line), so that the same arguments give the same files")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


_T0 = time.time()


def phase(msg):
    """Rank-0 progress line on stderr (wall clock since start): where a slow launch spends its time."""
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench %7.1fs] %s" % (time.time() - _T0, msg), file=sys.stderr, flush=True)


WORKLOAD = ("LSUN Cats 256^2 train.py step (StyleGAN2-256 generator + unimodal similarity+flow STN @128, perceptual VGG16 loss, "
            "Adam, EMA), synthetic latents + seeded random weights")


def workload_config(args, dtype="f32"):
    return {"workload": WORKLOAD + (" -- BASELINE config 2 (fp32)" if dtype == "f32" else
                                    " -- BASELINE config 3 (bf16 activations, fp32 master weights / accumulation)"),
            "step_mode": "eager" if args.no_graph else "whole-step CUDA graph replay",
            "per_gpu_batch": args.batch, "global_batch": args.batch * args.gpus, "gen_size": 256, "flow_size": 128,
            "parallelism": "dp%d" % args.gpus, "activation_layout": "NHWC (channels-last) generator + STN trunk",
            "l2_policy": "inputs larger than L2 (activations of one step >> 126 MB)",
            "cudnn": "deterministic (heuristic choice)" if args.dump_outputs else "benchmark (timed choice)"}


# --------------------------------------------------------------------------------------------------- reference arm
def cpu_threads():
    """All host cores, capped at 64: beyond that ATen's intra-op threading of these small convolutions gets slower."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("GG_CPU_THREADS", "64"))))


def cpu_step_rate(batch, steps=1, warmup=0):
    """The reference's training iteration on all host cores -> (images/s, s/step, kind).  kind "reference": the UNMODIFIED
    reference code (oracle/_ref/refpy_cpu, byte-compiled from /root/reference by oracle/build_ref.py) through its own native
    CPU branches (oracle/reference_step.py); kind "port": the oracle port (this repo's host code on the oracle's CPU op
    set) when that tree was not built."""
    import contextlib
    from oracle import reference_step
    if reference_step.available() and os.environ.get("GG_CPU_KIND", "reference") == "reference":
        with contextlib.redirect_stdout(sys.stderr):   # the reference prints ("Loading VGG ..."); stdout carries ONE JSON line
            rate, sec, _ = reference_step.step_rate(batch, steps=steps, warmup=warmup, threads=cpu_threads())
        return rate, sec, "reference"
    from oracle import opset
    from gangealing_b200.training import TrainConfig, Trainer
    torch.set_num_threads(cpu_threads())
    cfg = TrainConfig(batch=batch)
    tr = Trainer(cfg, "cpu", ops=opset.cpu_ops())
    for _ in range(warmup):
        tr.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = tr.step()
    float(out["p"].detach())
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, "port"


def run_reference(args):
    """The reference algorithm on the host cores.  The line reports what THIS arm ran (CPU, eager, NCHW, a bounded per-step
    batch), not the GPU arm's configuration; --steps / --warmup are honoured up to a wall-clock bound (each CPU step of
    batch 2 takes 5-20 s), and the clamp is stated."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    cores = cpu_threads()
    max_steps = int(os.environ.get("GG_CPU_MAX_STEPS", "6"))
    steps = max(1, min(args.steps, max_steps))
    warm = max(0, min(args.warmup, 1))
    rate, sec, kind = cpu_step_rate(args.cpu_batch, steps=steps, warmup=warm)
    sample = "%d step(s) of per-step batch %d (a bounded sample of the %d-per-GPU workload), %d host threads" % (
        steps, args.cpu_batch, args.batch, cores)
    cfg = {"workload": WORKLOAD + " -- BASELINE config 2 (fp32)", "step_mode": ("eager, CPU: the unmodified reference code (train.py:106-136 over oracle/_ref/refpy_cpu)" if kind == "reference"
                         else "eager, CPU (reference algorithm, oracle port)"),
           "per_step_batch": args.cpu_batch, "gen_size": 256, "flow_size": 128, "parallelism": "none (rank 0 host cores)",
           "activation_layout": "NCHW", "host_threads": cores,
           "steps_requested": args.steps, "warmup_requested": args.warmup,
           "clamp": "steps <= %d, warmup <= 1: a CPU step takes seconds; the sample is bounded to keep the run within minutes" % max_steps}
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------- our arm
DUMP_SAMPLE = 1 << 20   # parameters kept per module by snapshot(): 4 MB of float32 each


def snapshot(tr, out):
    """What the last timed step computed, copied to the host: the losses step() returned and the STN's parameters and their
    EMA after its optimiser update -- all of them, or a fixed, seeded sample of DUMP_SAMPLE elements (the same positions in
    every run of the same configuration)."""
    arrays = {"loss_" + k: v.detach().double().cpu().numpy().reshape(-1) for k, v in out.items()}
    for name, module in (("stn_params", tr.t_module), ("stn_ema_params", tr.t_ema)):
        flat = torch.cat([p.detach().float().reshape(-1) for p in module.parameters()])
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            flat = flat[idx.to(flat.device)]
        arrays[name] = flat.cpu().numpy()
    return arrays


def measure(args, dtype, dev, rank, world, distributed, want_clocks, want_outputs=False):
    """Build the trainer for `dtype`, warm up, probe the roofline kernel, capture the step, time `args.steps` steps twice
    (device-resident latents; end to end with host latents) -> dict of raw measurements (max over ranks)."""
    import torch.distributed as dist
    from gangealing_b200 import _lib
    from gangealing_b200.op import nhwc as nhwc_ops
    from gangealing_b200.op import styled_tail
    from gangealing_b200.training import TrainConfig, Trainer

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = TrainConfig(batch=args.batch, dtype=dtype, grad_compression=os.environ.get("GG_GRAD_COMPRESSION", "bf16" if dtype == "bf16" else "none"),
                      bucket_cap_mb=int(os.environ.get("GG_BUCKET_MB", "25")))
    tr = Trainer(cfg, dev, distributed=distributed)
    phase("trainer built (%s)" % dtype)

    def sync_all():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        tr.step()
    sync_all()
    phase("eager warm-up done")

    # ---- roofline probe: the dominant hand-written kernel (fused blur+noise+bias+lrelu tail) timed with CUDA
    #      events on its launching stream, inside real training steps of this workload (eager, so that the events
    #      bracket individual launches; a CUDA graph replay offers no per-kernel events)
    styled_tail.TIMING = []        # NCHW fused tail (not used by the channels-last pipeline)
    nhwc_ops.TIMING = styled_tail.TIMING
    calls0 = _lib.CALLS
    probe_steps = 2
    for _ in range(probe_steps):
        tr.step()
    sync_all()
    calls_per_step = (_lib.CALLS - calls0) // probe_steps
    timing, styled_tail.TIMING, nhwc_ops.TIMING = styled_tail.TIMING, None, None

    if not args.no_graph:
        tr.capture(warmup=2)   # a capture failure is an error: the bench never silently measures a different mode
        phase("step captured as a CUDA graph")
        for _ in range(2):
            tr.step()
        sync_all()

    # ---- timed region 1: device-resident inputs (latents drawn on the device, like reference loss.py:24)
    sampler = ClockSampler(local_rank) if (rank == 0 and want_clocks) else None
    if sampler:
        sampler.start()
    st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    profile = os.environ.get("GG_PROFILE") == "1"   # `ncu --profile-from-start off`: capture the timed steps only
    if profile:
        torch.cuda.cudart().cudaProfilerStart()
    st.record()
    for _ in range(args.steps):
        out = tr.step()
    en.record()
    sync_all()
    if profile:
        torch.cuda.cudart().cudaProfilerStop()
    ms = st.elapsed_time(en)
    phase("timed region 1 done")
    outputs = snapshot(tr, out) if want_outputs else None
    if sampler:
        sampler.stop_flag.set()

    # ---- timed region 2: end to end through the public step() with HOST latents (pinned) and a host read of the loss
    z_host = torch.randn(args.batch, cfg.dim_latent).pin_memory()
    loss_host = torch.zeros(3).pin_memory()
    sync_all()
    st2, en2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st2.record()
    for _ in range(args.steps):
        z = z_host.to(dev, non_blocking=True)
        out = tr.step(z)
        loss_host.copy_(torch.stack([out["p"].detach().reshape(()), out["tv"].detach().reshape(()), out["f"].detach().reshape(())]))
        torch.cuda.current_stream().synchronize()  # the host now holds this step's losses
    en2.record()
    sync_all()
    ms2 = st2.elapsed_time(en2)

    t = torch.tensor([ms, ms2], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms2 = t.tolist()
    return {"tr": tr, "cfg": cfg, "ms": ms, "ms2": ms2, "timing": timing, "calls": calls_per_step * args.steps, "outputs": outputs,
            "clocks": sampler.summary() if sampler else None, "losses": {k: float(v.detach()) for k, v in out.items()}}


def roofline_of(m, args, dtype):
    """Roofline of the dominant hand-written kernel: the fused blur+noise+bias+act tail at the 256^2 layer."""
    timing = m["timing"]
    if not timing:
        return None
    peak, peak_src = peaks()
    biggest = max(t_[2] for t_ in timing)
    sel = [t_ for t_ in timing if t_[2] == biggest]
    durs = [a.elapsed_time(b) for a, b, _ in sel]
    avg_ms = sum(durs) / len(durs)
    achieved = biggest / (avg_ms * 1e-3) / 1e9
    kname = "blur_nhwc_kernel<%s, MODE=1 (fused tail), SEP=1> (channels-last blur+noise+bias+lrelu tail, 256^2 layer)" % (
        "float" if dtype == "f32" else "__nv_bfloat16")
    # DRAM bytes per launch of this kernel from a committed `ncu --set full` capture (same shape, batch and dtype only)
    traffic, traffic_src = None, None
    for name in ("r02_nhwc_b32_traffic_%s.json" % dtype, "r01_nhwc_b32_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("per_gpu_batch") == args.batch and tj.get("dtype", "f32") == dtype:
                for k, v in tj["kernels"].items():
                    if k.startswith("blur_nhwc_kernel") and v.get("fused_tail", True):
                        traffic = v.get("dram_bytes_per_launch")
                        traffic_src = "ncu --set full capture committed as profiles/%s (not measured by this run)" % name
                        break
            if traffic is not None:
                break
    return {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": biggest, "launches_timed": len(durs), "avg_launch_ms": avg_ms, "peak_source": peak_src}


def run_ours(args):
    import torch.distributed as dist
    from gangealing_b200.training import distributed as gdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")  # required for capturing NCCL work in CUDA graphs
        gdist.setup_distributed("nccl")
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    rank = gdist.get_rank()
    # a dump must be the same on every run with the same arguments: cuDNN's timed algorithm choice can differ from run to
    # run, and the training step carries any difference forward through Adam -- so a dumping run takes its heuristic
    # choice of deterministic algorithms (config.cudnn says which mode the timed numbers were measured in)
    torch.backends.cudnn.benchmark = not args.dump_outputs
    torch.backends.cudnn.deterministic = bool(args.dump_outputs)
    phase("process group ready (world %d)" % world)

    m = measure(args, args.dtype, dev, rank, world, distributed, want_clocks=True,
                want_outputs=bool(args.dump_outputs) and rank == 0)
    images = args.batch * world * args.steps
    extra = None
    other = "bf16" if args.dtype == "f32" else None
    if other and os.environ.get("GG_BENCH_EXTRA", "1") == "1" and not args.no_extra:
        # BASELINE config 3 (bf16 activations) measured in the same run, same box, same steps: reported under `config3_bf16`
        tr0 = m.pop("tr")
        tr0.release_graph()
        del tr0
        torch.cuda.empty_cache()
        try:
            m3 = measure(args, other, dev, rank, world, distributed, want_clocks=False)
        except Exception as exc:
            # the ADDITIONAL measurement must not take the headline line down -- on one GPU.  With several ranks a failure may
            # be one rank's alone: re-raise, so that torchrun ends the job instead of the other ranks waiting in a collective
            if distributed:
                raise
            m3, m["tr"] = None, None
            extra = {"metric": METRIC, "dtype": "bf16", "value": None, "unit": UNIT, "error": "%s: %s" % (type(exc).__name__, exc)}
            phase("config-3 measurement failed: %r" % (exc,))
        if m3 is not None:
            extra = {"metric": METRIC, "dtype": "bf16", "value": images / (m3["ms"] / 1e3), "unit": UNIT,
                     "ms_per_step": m3["ms"] / args.steps,
                     "e2e": {"value": images / (m3["ms2"] / 1e3), "unit": UNIT, "ms_per_step": m3["ms2"] / args.steps},
                     "config": workload_config(args, "bf16"), "roofline": roofline_of(m3, args, "bf16") if rank == 0 else None,
                     "gpu_launches": m3["calls"], "losses": m3["losses"], "grad_allreduce": m3["cfg"].grad_compression}
            m["tr"] = m3.pop("tr")
    tr = m["tr"]
    if rank != 0:
        finish(distributed, tr)
        return
    ms, ms2 = m["ms"], m["ms2"]
    value = images / (ms / 1e3)
    e2e = images / (ms2 / 1e3)
    cfg = m["cfg"]
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            rate, sec, kind = cpu_step_rate(args.cpu_batch, steps=1, warmup=0)
            cpu = {"value": rate, "unit": UNIT, "cores": cpu_threads(), "kind": kind,
                   "sample": "1 step of per-step batch %d on %d host threads of %d cores (%.1f s)" % (
                       args.cpu_batch, cpu_threads(), os.cpu_count(), sec)}
        except Exception as exc:  # the baseline must never take the bench down
            cpu = {"value": None, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": "failed: %r" % (exc,)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": workload_config(args, args.dtype),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": args.batch * cfg.dim_latent * 4 * world,
                    "d2h_bytes_per_step": 12 * world, "ms_per_step": ms2 / args.steps},
            "gpu_launches": m["calls"], "roofline": roofline_of(m, args, args.dtype), "cpu_baseline": cpu,
            "clocks": m["clocks"], "losses": m["losses"]}
    if extra is not None:
        line["config3_bf16"] = extra
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, array in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), array)
    print(json.dumps(line), flush=True)
    phase("result printed")
    finish(distributed, tr)
    phase("process group torn down")


def finish(distributed, tr):
    """Tear the process group down AFTER the result is out.  A watchdog ends the process with status 0 if NCCL's
    teardown stalls (communicators referenced by a captured graph have been seen to block in destroy)."""
    sys.stdout.flush()
    if not distributed:
        return
    import torch.distributed as dist
    watchdog = threading.Timer(20.0, lambda: os._exit(0))
    watchdog.daemon = True
    watchdog.start()
    try:
        dist.barrier()
        if tr is not None:
            tr.release_graph()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    finally:
        watchdog.cancel()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
