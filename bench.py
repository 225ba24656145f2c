#!/usr/bin/env python
"""Headline benchmark: volumes/sec of 3D-LDM DDPM sampling (BASELINE.json cfg4).

Workload (config.workload = "ddpm_3d_ldm_sampling"): UNet3DModelWithAttention(in=3, base 128,
mults (1,2,4), time_emb 256, groups 8, heads 4) on 3x40x48x40 latents, cosine schedule,
T = 1000 reverse steps per volume, random-init weights, synthetic latents.

A "step" = one reverse step (UNet forward + fused DDPM update) over this rank's batch of
volumes.  value = (volumes in flight over all ranks) / (T * seconds per step): every reverse
step does identical work, so timing K consecutive steps of a real trajectory (t = T-1, T-2, ...)
measures the loop; `--steps 1000` times complete volumes.  Sampling shards the batch across
ranks with no communication (scaling = "weak": per-GPU batch fixed).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference]
                  [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...            (one rank per GPU; rank 0 prints ONE JSON line)

--impl reference times the reference's own algorithm for the same path on the host CPU cores
(the oracle port of the reference modules, all threads; /root/reference does not exist on the
GPU box and a Python reference cannot be compiled into oracle/_ref).
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS = 1000
LATENT = (3, 40, 48, 40)
MODEL_KW = dict(in_channels=3, base_channels=128, channel_mults=(1, 2, 4), time_emb_dim=256,
                groups=8, num_heads=4)
CONV_FLOPS_PER_SAMPLE = 1273.4e9  # SURVEY.md 8(d): conv part of one UNet forward at cfg4


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": d.get("bf16_tflops_sustained", 1371.0), "hbm": d.get("hbm_gbs", 6555.2),
                "source": "measured"}
    return {"tflops": 1590.0, "hbm": 6650.0, "source": "fallback"}


def load_traffic(batch: int):
    """DRAM bytes per step of the two kernel families, from the committed `ncu` capture of this very
    command (profiles/*_step_dram_traffic.json; the capture's command line is in its "source").
    None when no capture matches the batch size -- a number measured under a profiler is never
    produced at bench time."""
    import glob
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_step_dram_traffic.json")), reverse=True):
        try:
            d = json.load(open(f))
        except Exception:  # noqa: BLE001
            continue
        if d.get("batch_per_gpu") == batch:
            d["file"] = os.path.relpath(f, ROOT)
            return d
    return None


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML DURING the timed region."""

    def __init__(self, index: int, period_s: float = 0.05):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(self.h))
                for n, bit in names.items():
                    if mask & bit:
                        self.reasons.add(n)
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            time.sleep(self.period)

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        sm = sorted(self.sm)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(sm)}
        if self.err:
            out["error"] = self.err
        return out


# ------------------------------------------------------------------------------------------
def cpu_reference_rate(n_forwards: int, threads: int):
    """Reference algorithm (oracle port) on the host cores: seconds per reverse step at B = 1."""
    import torch
    from oracle import reference_oracle as O
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
        UNet3DModelWithAttention
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    sd = {k: v.detach() for k, v in UNet3DModelWithAttention(**MODEL_KW).state_dict().items()}
    buf = O.schedule_buffers(O.cosine_betas(T_STEPS))
    x = torch.randn(1, *LATENT)
    times = []
    first = None
    with torch.no_grad():
        for i in range(n_forwards + 1):
            t = torch.full((1,), T_STEPS - 1 - i, dtype=torch.long)
            t0 = time.perf_counter()
            eps = O.unet3d_forward(sd, x, t)
            if first is None:     # the checker's answer for one (x, t): parity_record() compares the device paths
                first = (sd, x.clone(), t.clone(), eps.clone())
            x = O.p_sample_update(buf, x, t, eps, torch.randn_like(x))
            times.append(time.perf_counter() - t0)
    return sum(times[1:]) / n_forwards, first  # first call = warm-up


def parity_record(torch, dev, first):
    """Noise prediction of the device paths against the fp32 CPU oracle on the SAME weights and
    input (B = 1, full latent): the default bf16 path and the split precision mode (DESIGN 3.4),
    plus what one reverse step costs in each at B = 1."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
        UNet3DModelWithAttention
    sd, x, t, want = first
    model = UNet3DModelWithAttention(**MODEL_KW)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    diff = quiet(GaussianDiffusionLatent3D, model, LATENT[0], timesteps=T_STEPS).to(dev)
    out = {"what": "eps rel-L2 against the fp32 CPU oracle, B = 1, t = %d, same weights and input" % int(t[0]),
           "tolerance": {"bf16": 2e-2, "split": 3e-4}}
    xd, td = x.to(dev), t.to(dev)
    with torch.no_grad():
        for prec in ("bf16", "split"):
            model.precision = prec
            got = model(xd, td)
            err = ((got.cpu() - want).norm() / want.norm()).item()
            for _ in range(3):
                diff.p_sample(xd, td)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(5):
                diff.p_sample(xd, td)
            e1.record()
            torch.cuda.synchronize(dev)
            out[prec] = {"eps_rel_l2": err, "reverse_step_ms_b1": e0.elapsed_time(e1) / 5}
    del diff, model
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    n = max(1, args.steps)
    w = max(1, args.warmup)
    # bounded sample: `steps` timed reverse steps at B = 1 after `warmup` untimed ones
    from oracle import reference_oracle as O
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
        UNet3DModelWithAttention
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    sd = {k: v.detach() for k, v in UNet3DModelWithAttention(**MODEL_KW).state_dict().items()}
    buf = O.schedule_buffers(O.cosine_betas(T_STEPS))
    x = torch.randn(1, *LATENT)
    n = min(n, 5)
    w = min(w, 1)
    t_total = 0.0
    with torch.no_grad():
        for i in range(w + n):
            t = torch.full((1,), T_STEPS - 1 - i, dtype=torch.long)
            t0 = time.perf_counter()
            x = O.p_sample_update(buf, x, t, O.unet3d_forward(sd, x, t), torch.randn_like(x))
            if i >= w:
                t_total += time.perf_counter() - t0
    sec_per_step = t_total / n
    value = 1.0 / (T_STEPS * sec_per_step)
    sample = f"{n} reverse steps at batch 1 after {w} warm-up, extrapolated x{T_STEPS // 1} per volume"
    line = {
        "impl": "reference", "metric": "volumes/sec (3D LDM DDPM sampling)", "value": value,
        "unit": "volumes/s", "n_gpus": args.gpus, "steps": n, "warmup": w,
        "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ddpm_3d_ldm_sampling", "latent": list(LATENT), "timesteps": T_STEPS,
                   "model": "UNet3DModelWithAttention(base 128, mults 1-2-4)", "batch_per_step": 1,
                   "device": "host CPU"},
        "cpu_baseline": {"value": value, "unit": "volumes/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
def family_times(torch, dev, seq, plain_graph, reps: int = 5, load_replays: int = 4):
    """Per-family kernel time of ONE reverse step measured INSIDE a replayed CUDA graph.

    `seq` = [(family, fn)] is the step's launch list.  The step is captured once more with an
    external timing event (an event-record node) at every boundary between two families;
    consecutive events bracket contiguous runs of one family, so the family sums telescope to the
    instrumented step's duration by construction (sum <= step).  Each sample is taken right after
    `load_replays` replays of the plain step graph so that clocks / power state are those of the
    timed loop.  Falls back to one small graph per run with ordinary events between the graphs
    if external events cannot be captured."""
    fams = [f for f, _ in seq]
    bounds = [0] + [i for i in range(1, len(seq)) if fams[i] != fams[i - 1]] + [len(seq)]
    runs = [(fams[a], a, b) for a, b in zip(bounds, bounds[1:])]
    acc = {}
    steps = []
    mode = "event-record nodes inside one graph"
    try:
        evs = []
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(dev)
        with torch.cuda.graph(g):
            for fam, a, b in runs:
                e = torch.cuda.Event(enable_timing=True, external=True)
                e.record()
                evs.append(e)
                for _, fn in seq[a:b]:
                    fn()
            e = torch.cuda.Event(enable_timing=True, external=True)
            e.record()
            evs.append(e)
        for _ in range(reps):
            for _ in range(load_replays):
                plain_graph.replay()
            g.replay()
            torch.cuda.synchronize(dev)
            for (fam, _, _), e0, e1 in zip(runs, evs, evs[1:]):
                acc[fam] = acc.get(fam, 0.0) + e0.elapsed_time(e1)
            steps.append(evs[0].elapsed_time(evs[-1]))
    except Exception as exc:  # noqa: BLE001
        mode = f"one graph per run, events between graph launches ({type(exc).__name__})"
        acc, steps = {}, []
        torch.cuda.synchronize(dev)
        graphs = []
        for fam, a, b in runs:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _, fn in seq[a:b]:
                    fn()
            graphs.append(g)
        for _ in range(reps):
            for _ in range(load_replays):
                plain_graph.replay()
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(runs) + 1)]
            evs[0].record()
            for g, e in zip(graphs, evs[1:]):
                g.replay()
                e.record()
            torch.cuda.synchronize(dev)
            for (fam, _, _), e0, e1 in zip(runs, evs, evs[1:]):
                acc[fam] = acc.get(fam, 0.0) + e0.elapsed_time(e1)
            steps.append(evs[0].elapsed_time(evs[-1]))
    out = {k: v / reps for k, v in acc.items()}
    return out, sum(steps) / len(steps), (max(steps) - min(steps)) / (sum(steps) / len(steps)), mode, len(runs)


def gpu_comparator(torch, dev, B: int, sd):
    """SURVEY.md 8(d) "GPU comparator": the reference's own PyTorch graph (the oracle restatement:
    the same ATen / cuDNN / cuBLAS calls the reference modules make) run EAGERLY on this GPU at
    the benched shape -- fp32 with TF32 (train.py:72) and under autocast(bf16) (train.py:395),
    cudnn.benchmark on (train.py:71).  A reported baseline like cpu_baseline; nothing of it is on
    the product path."""
    from oracle import reference_oracle as O
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
           torch.get_float32_matmul_precision())
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = True
    torch.set_float32_matmul_precision("high")
    out = {"cudnn": torch.backends.cudnn.version(), "batch_per_step": B,
           "what": "reference graph (oracle restatement) eager on the same GPU, one reverse step"}
    try:
        buf = {k: v.to(dev) for k, v in O.schedule_buffers(O.cosine_betas(T_STEPS)).items()}
        x = torch.randn(B, *LATENT, device=dev)
        t = torch.full((B,), 500, device=dev, dtype=torch.long)

        def step(autocast):
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
            with torch.no_grad():
                with ctx:
                    eps = O.unet3d_forward(sd, x, t)
                return O.p_sample_update(buf, x, t, eps.float(), torch.randn_like(x))

        for name, ac in (("autocast_bf16", True), ("tf32", False)):
            for _ in range(2):
                step(ac)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(3):
                step(ac)
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / 3
            out[name] = {"ms_per_step": ms, "value": B / (T_STEPS * ms * 1e-3), "unit": "volumes/s",
                         "tflops": B * 1276.4e9 / (ms * 1e-3) / 1e12}
    except Exception as exc:  # noqa: BLE001
        out["error"] = repr(exc)
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32 = old[0], old[1]
        torch.set_float32_matmul_precision(old[2])
        torch.cuda.empty_cache()
    return out


def train_record(args, torch, dist, rank, world, dev, B: int, K: int, W: int):
    """BASELINE.json cfg5: K timed DDP training steps of the 3D LDM UNet at B latents per GPU --
    q_sample (noise drawn in-kernel) + forward + min-SNR loss + backward with the bucketed NCCL
    all-reduce overlapped (ddpm_3d_ldm/train.py:232-233,395-400) + fused Adam.  Returns the
    record that goes on the bench line (rank 0) or None."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
        UNet3DModelWithAttention
    from mri_image_generation_b200.parallel import wrap_ddp

    torch.manual_seed(0)
    model = UNet3DModelWithAttention(**MODEL_KW).to(dev).train()
    overlap = not getattr(args, "torch_ddp", False)
    # --no-ddp (attribution only): N independent replicas, no gradient exchange -- what the box
    # itself costs when all N GPUs train at once (shared power / thermal envelope), to be
    # subtracted from the DDP step before blaming the all-reduce
    replicas_only = bool(getattr(args, "no_ddp", False))
    net = wrap_ddp(model, dev, overlap=overlap) if (world > 1 and not replicas_only) else model
    diff = quiet(GaussianDiffusionLatent3D, net, LATENT[0], timesteps=T_STEPS).to(dev)
    if getattr(args, "torch_adam", False):
        opt = torch.optim.Adam(model.parameters(), lr=2e-4)
    else:  # one-launch Adam (mri_adam_step), same update rule and state layout
        from mri_image_generation_b200.optim import Adam
        opt = Adam(model.parameters(), lr=2e-4)
    torch.manual_seed(1234 + rank)
    z = torch.randn(B, *LATENT, device=dev)

    def step():
        t = torch.randint(1, T_STEPS, (B,), device=dev)
        opt.zero_grad(set_to_none=True)
        loss = diff.p_losses(z, t, cond=None, min_snr_gamma=5.0)
        loss.backward()
        opt.step()
        return loss

    def timed(n):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            loss = step()
        e1.record()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        return e0.elapsed_time(e1), loss

    for _ in range(max(W, 4)):   # two eager steps, the capturing one, a replayed one
        step()
    sampler = ClockSampler(dev.index) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_dev, loss = timed(K)
    clocks = sampler.stop() if sampler else None
    # end to end: every step's latents come from pinned host memory and every step's loss is read
    # back to the host (a 4-byte D2H that also synchronises the step)
    z_host = z.cpu().pin_memory()
    Ke = min(K, 10)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(Ke):
        z.copy_(z_host, non_blocking=True)
        loss_host = step().item()
    e1.record()
    torch.cuda.synchronize(dev)
    ms_e2e = e0.elapsed_time(e1)
    # ---- communication: per-bucket events, exposed time, overlap on / off --------------------
    comm = None
    ms_noov = 0.0
    prog = model.program(B, LATENT[1:], training=True)
    if world > 1 and overlap and not replicas_only:
        gs = net.grad_sync
        gs.time_buckets = True
        reports = []
        for _ in range(3):
            step()
            torch.cuda.synchronize(dev)
            reports.append(gs.bucket_report())
        gs.time_buckets = False
        comm = reports[-1]
        if comm is not None:
            comm["exposed_comm_ms_samples"] = [r["exposed_comm_ms"] for r in reports if r]
            comm["n_buckets"] = len(gs.buckets_last_step)
            comm["bucket_cap_mb"] = gs.bucket_bytes / (1 << 20)
        # A/B: one bucket = the all-reduce starts after the whole backward (no overlap)
        cap = gs.bucket_bytes
        gs.bucket_bytes = 1 << 40
        prog.bwd_segments = []
        for _ in range(4):
            step()
        ms_noov, _ = timed(min(K, 10))
        ms_noov /= min(K, 10)
        gs.bucket_bytes = cap
        prog.bwd_segments = []
    ms = torch.tensor([ms_dev, ms_e2e, ms_noov], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    ms_per_step = ms[0].item() / K
    ms_e2e_step = ms[1].item() / Ke
    flops = B * 3 * 1276.4e9  # fwd + bwd = 3 x fwd (SURVEY.md 8d: 30.62 TFLOP per 8-sample step)
    peaks = load_peaks()
    rec = {
        "metric": "training samples/sec (3D LDM UNet DDP step)", "value": world * B / (ms_per_step / 1e3),
        "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": max(W, 4), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "ddpm_3d_ldm_train_step", "latent": list(LATENT), "batch_per_gpu": B,
                   "model": "UNet3DModelWithAttention(base 128, mults 1-2-4, 136.4M params)",
                   "step": "q_sample (in-kernel Philox) + fwd + min-SNR loss + bwd + DDP all-reduce + Adam",
                   "ddp": ("none (1 GPU)" if world == 1 else "NONE: independent replicas (--no-ddp, attribution run)"
                           if replicas_only else "torch DDP (reducer after backward)" if not overlap
                           else "bucketed NCCL all-reduce (545.6 MB fp32) overlapped with the backward launch list"),
                   "optimizer": "torch.optim.Adam" if getattr(args, "torch_adam", False) else "mri_b200 fused Adam",
                   "loss": float(loss.item())},
        "e2e": {"value": world * B / (ms_e2e_step / 1e3), "unit": "samples/s",
                "h2d_bytes_per_step": z_host.numel() * 4, "d2h_bytes_per_step": 4, "steps": Ke,
                "path": "pinned host latents -> p_losses -> backward -> Adam -> loss.item() on the host, every step",
                "last_loss": loss_host},
        # launches of this library per step: forward + backward launch lists (replayed as CUDA
        # graphs), q_sample, loss forward / backward, weight re-pack, gradient finalisation, Adam
        "gpu_launches": (len(prog.ops) + len(prog.bwd_ops) + 8) * K,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": flops / (ms_per_step * 1e-3) / 1e12,
                     "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": flops / (ms_per_step * 1e-3) / 1e12 / peaks["tflops"],
                     "note": "whole step (all kernels + optimizer + all-reduce), algorithmic conv+attention FLOPs",
                     "executed_gemm_flops": prog.gemm_flops + prog.bwd_flops},
    }
    if comm is not None:
        rec["comm"] = comm
        rec["no_overlap_ms_per_step"] = ms[2].item()
        rec["overlap_gain_ms"] = ms[2].item() - ms_per_step
    del opt, diff, net, model
    torch.cuda.empty_cache()
    return rec


# ------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from mri_image_generation_b200 import _lib, ops
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
        UNet3DModelWithAttention

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.require_device()
    B, K, W = args.batch, args.steps, max(3, args.warmup)

    torch.manual_seed(0)  # identical random-init weights on every rank
    model = UNet3DModelWithAttention(**MODEL_KW).to(dev).eval()
    diff = quiet(GaussianDiffusionLatent3D, model, LATENT[0], timesteps=T_STEPS).to(dev)
    torch.manual_seed(1234 + rank)
    prog = model.program(B, LATENT[1:])
    x_T = torch.randn(B, *LATENT, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing: K replays of the captured reverse step --------------------
    with torch.no_grad():
        diff._reverse_loop(prog, x_T, T_STEPS - 1, W, "ddpm")  # builds + captures + W warm-up steps
        graph = prog._step_graphs["ddpm"][2]
        prog.x_in.copy_(x_T)
        prog.t_in.fill_(T_STEPS - 1)
        sampler = ClockSampler(local_rank)
        barrier()
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            if i and i % T_STEPS == 0:   # the trajectory reached t = 0: the next volume starts at T - 1
                prog.t_in.fill_(T_STEPS - 1)
            graph.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        finite = bool(torch.isfinite(prog.x_in).all().item())
        x_last = prog.x_in.cpu() if args.dump_outputs and rank == 0 else None   # x_{t-1} of step K

        # ---- end to end through the public API with host buffers, every step ---------------
        # Every step's input comes from pinned host memory and every step's result goes back to
        # pinned host memory, all inside the timed region.  The copies run on two copy streams so
        # that the H2D of step i + 1 and the D2H of step i - 1 overlap the compute of step i (the
        # steps of this loop are independent requests; a dependent loop keeps its state on the device).
        x_host = torch.randn(B, *LATENT).pin_memory()
        out_host = torch.empty(B, *LATENT).pin_memory()
        x_devs = [torch.empty(B, *LATENT, device=dev) for _ in range(2)]
        Ke = min(K, 20)
        cur = torch.cuda.current_stream(dev)
        copy_in, copy_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        for i in range(2):
            diff.p_sample(x_devs[0].copy_(x_host, non_blocking=True),
                          torch.full((B,), T_STEPS - 1 - i, device=dev, dtype=torch.long))
        barrier()

        def h2d(b):
            with torch.cuda.stream(copy_in):
                copy_in.wait_event(ev_free[b])      # the step that last read this buffer is done
                x_devs[b].copy_(x_host, non_blocking=True)
                ev_in[b].record(copy_in)

        e0.record()
        for b in range(2):
            ev_free[b].record(cur)
        copy_in.wait_stream(cur)                    # nothing is copied before the timer starts
        copy_out.wait_stream(cur)
        h2d(0)
        for i in range(Ke):
            b = i & 1
            if i + 1 < Ke:
                h2d(1 - b)
            cur.wait_event(ev_in[b])
            t = torch.full((B,), T_STEPS - 1 - i, device=dev, dtype=torch.long)
            y = diff.p_sample(x_devs[b], t)
            ev_free[b].record(cur)
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(copy_out):
                copy_out.wait_event(done)
                out_host.copy_(y, non_blocking=True)
            y.record_stream(copy_out)
        cur.wait_stream(copy_out)                   # the last result has reached the host
        e1.record()
        torch.cuda.synchronize(dev)
        ms_e2e = e0.elapsed_time(e1)

        # ---- per-family kernel time, measured INSIDE the replayed step graph ------------------
        from mri_image_generation_b200 import ops as _ops
        gemm_idx = [i for i, n in enumerate(prog.op_names) if n.startswith("gemm:")]
        gn_idx = {i for i, _ in prog.gn_ops}   # GroupNorm-apply launches: the HBM-bound family
        gemm_set = set(gemm_idx)
        rng = diff._rng(dev)
        inc = _ops.randn_offset_increment(prog.x_in.numel())
        seq = [("other", lambda: _ops.memset_zero(prog._arena, max(prog._arena_used, 4) * 8))]
        fh = prog.fused_head if os.environ.get("MRI_FUSED_STEP", "1") != "0" else None
        for i, fn in enumerate(prog.ops[:-1] if fh is not None else prog.ops):
            tc = i in gemm_set or prog.op_names[i].startswith(("attn:", "tc:"))   # tcgen05 kernels
            seq.append(("gemm" if tc else "gn" if i in gn_idx else "other", fn))
        if fh is not None:   # out_conv's tap sum + DDPM update (in-kernel Philox) in one launch
            seq.append(("other", lambda: _ops.tap_gather_step(
                fh["y"], fh["bias"], prog.B, fh["D"], fh["H"], fh["W"], fh["ndim"], fh["cout"], fh["ldy"],
                prog.x_in, 0, rng=rng, t=prog.t_in, betas=diff.betas,
                sqrt_1mac=diff.sqrt_one_minus_alphas_cumprod, sqrt_recip_alphas=diff.sqrt_recip_alphas,
                post_var=diff.posterior_variance)))
        else:
            seq.append(("other", lambda: _ops.ddpm_step_rng(
                prog.x_in, prog.eps_nhwc, rng, prog.t_in, diff.betas, diff.sqrt_one_minus_alphas_cumprod,
                diff.sqrt_recip_alphas, diff.posterior_variance, prog.x_in, eps_nhwc_ldc=prog.cout_pad,
                channels=prog.cout)))
        seq.append(("other", lambda: _ops.step_advance(prog.t_in, -1, rng=rng, rng_increment=inc)))
        prog.x_in.copy_(x_T)
        prog.t_in.fill_(T_STEPS - 1)
        fam, inst_ms, inst_spread, fam_mode, n_runs = family_times(torch, dev, seq, graph)
        gemm_ms, gn_ms, other_ms = fam.get("gemm", 0.0), fam.get("gn", 0.0), fam.get("other", 0.0)
        gn_bytes = sum(nb for _, nb in prog.gn_ops)
        evs = []
        if args.per_op:   # eager per-op events (each launch bracketed on its own): --per-op only
            reps = 3
            stream = torch.cuda.current_stream(dev)
            for r in range(reps + 1):
                _ops.memset_zero(prog._arena, max(prog._arena_used, 4) * 8)
                for i, fn in enumerate(prog.ops):
                    if i in gemm_idx and r > 0:
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record(stream)
                        fn()
                        b.record(stream)
                        evs.append((a, b))
                    else:
                        fn()
            torch.cuda.synchronize(dev)
        if args.per_op and rank == 0:
            per = {}
            for j, (a, b) in enumerate(evs):
                per.setdefault(gemm_idx[j % len(gemm_idx)], []).append(a.elapsed_time(b))
            rows = []
            for i, pl in zip(gemm_idx, prog.plans):
                msi = sum(per[i]) / len(per[i])
                rows.append((prog.op_names[i], msi, pl.flops / (msi * 1e-3) / 1e12, pl.grid(), pl.block_n,
                             pl.n_kb, pl.box, pl._args.sched))
            with open(args.per_op, "w") as f:
                for r_ in rows:
                    f.write("%-34s %8.3f ms %8.1f TF/s grid %6d bn %3d n_kb %4d box %s sched %d\n" % r_)

    t_ms = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t_ms.tolist()
    comparator = None
    if world == 1 and not args.no_gpu_comparator:
        sd_dev = {k: v.detach() for k, v in model.state_dict().items()}
        comparator = gpu_comparator(torch, dev, B, sd_dev)
    # ---- secondary record: BASELINE cfg5 DDP training step on the same N GPUs --------------------
    train = None
    if not args.no_train:
        train = train_record(args, torch, dist, rank, world, dev, args.train_batch,
                             min(K, args.train_steps), W)
    if rank != 0:
        return

    ms_per_step = ms / K
    value = world * B / (T_STEPS * ms_per_step / 1e3)
    e2e_val = world * B / (T_STEPS * (ms_e2e / Ke) / 1e3)
    peaks = load_peaks()
    # algorithmic FLOPs of one step: SURVEY.md 8(d) figure for the reference graph (conv 1273.4 G +
    # attention bmm 2.95 G per sample), not the padded shapes the kernel executes
    conv_flops = B * 1276.4e9
    executed_flops = prog.gemm_flops
    achieved = conv_flops / (gemm_ms * 1e-3) / 1e12
    x_bytes = x_host.numel() * 4
    # forward launch list (its last launch replaced by the fused gather + DDPM update) + step advance
    launches_per_step = len(prog.ops) + (1 if prog.fused_head is not None else 2)
    cpu = None
    parity = None
    if world == 1 or rank == 0:
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            nfw = 3
            sec, first = cpu_reference_rate(nfw, threads)
            cpu = {"value": 1.0 / (T_STEPS * sec), "unit": "volumes/s", "cores": threads,
                   "kind": "port",
                   "sample": f"{nfw} reverse steps at batch 1 ({sec:.2f} s each) x {T_STEPS} per volume"}
            if world == 1:
                parity = parity_record(torch, dev, first)
    traffic = load_traffic(B) or {}
    tr_gemm, tr_gn = traffic.get("gemm_tc", {}), traffic.get("gn_apply", {})
    line = {
        "metric": "volumes/sec (3D LDM DDPM sampling)", "value": value, "unit": "volumes/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "ddpm_3d_ldm_sampling", "latent": list(LATENT), "timesteps": T_STEPS,
                   "model": "UNet3DModelWithAttention(base 128, mults 1-2-4, 136.4M params)",
                   "batch_per_gpu": B, "parallelism": f"batch-sharded x{world}, no collective",
                   "l2": "per-step working set (273 MB bf16 weights + activations) exceeds the 126 MB L2",
                   "step": "one reverse step (UNet fwd + fused DDPM update) in a replayed CUDA graph",
                   "outputs_finite": finite},
        "e2e": {"value": e2e_val, "unit": "volumes/s", "h2d_bytes_per_step": x_bytes,
                "d2h_bytes_per_step": x_bytes, "steps": Ke,
                "path": "pinned host x_t -> GaussianDiffusionLatent3D.p_sample -> pinned host x_{t-1}; "
                        "copies on two copy streams, double-buffered against the compute stream"},
        "gpu_launches": launches_per_step * K,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 implicit GEMM: every convolution) + thin_in_conv_kernel + attn_flash_kernel (tcgen05 first convolution / fused attention)",
                     "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tflops"], "traffic": tr_gemm.get("dram_bytes"),
                     "traffic_note": ("DRAM bytes read + written by the %d GEMM launches of one step, ncu capture %s"
                                      % (tr_gemm.get("launches_per_step", 0), traffic.get("file"))) if tr_gemm else None,
                     "peak_source": peaks["source"] + " (bf16_tflops_sustained)",
                     "flops_per_step": conv_flops, "executed_flops_per_step": executed_flops,
                     "kernel_ms_per_step": gemm_ms,
                     "share_of_step": gemm_ms / inst_ms,
                     "timing": {"how": "CUDA events at every family boundary INSIDE one replayed step graph ("
                                       + fam_mode + "), mean of 5 samples each taken after 4 plain replays",
                                "instrumented_step_ms": inst_ms, "plain_step_ms": ms_per_step,
                                "spread": inst_spread, "event_pairs_per_step": n_runs,
                                "families_ms": {"gemm_tc": gemm_ms, "gn_apply": gn_ms, "other": other_ms}}},
        # second kernel family of the step: GroupNorm-apply (+SiLU, + time-embedding add, + residual),
        # HBM-bound; algorithmic bytes = 2 B read + 2 B written per element (+2 B with a residual)
        "roofline_hbm": {"bound": "hbm", "kernel": "gn_apply_kernel (all GroupNorm+SiLU launches of the step)",
                         "achieved": gn_bytes / (gn_ms * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": gn_bytes / (gn_ms * 1e-3) / 1e9 / peaks["hbm"],
                         "traffic": tr_gn.get("dram_bytes"),
                         "bytes_per_step": gn_bytes, "kernel_ms_per_step": gn_ms,
                         "share_of_step": gn_ms / inst_ms, "launches_per_step": len(prog.gn_ops)},
        "cpu_baseline": cpu,
    }
    if parity is not None:
        line["parity"] = parity
    if comparator is not None:
        line["gpu_comparator"] = comparator
    if train is not None:
        line["train"] = train
    if x_last is not None:
        dump_outputs(args.dump_outputs, {"x_prev": x_last})
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays) -> None:
    """--dump-outputs: every array as <out_dir>/<name>.npy in float32, for comparing two builds
    output for output.  Over DUMP_LIMIT_BYTES in all, only the leading samples (dim 0) that fit
    are written."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    for name, a in arrays.items():
        a = a.detach().float()
        if total > DUMP_LIMIT_BYTES:
            a = a[:max(1, a.shape[0] * DUMP_LIMIT_BYTES // total)]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def run_train(args, rank, world, local_rank):
    """Secondary workload (BASELINE.json cfg5) on its own: `--mode train` prints the training
    record (samples/s) as the line; the default sampling run carries the same record under
    "train"."""
    import torch
    import torch.distributed as dist
    from mri_image_generation_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.require_device()
    rec = train_record(args, torch, dist, rank, world, dev, args.batch, args.steps, max(3, args.warmup))
    if rank == 0:
        print(json.dumps(rec), flush=True)


def run_vae(args, rank, world, local_rank):
    """Secondary workload (SURVEY.md 8f row 1): VAE3D(4, 32, 3, latent 3) encode_to_latent of
    4x160x192x160 volumes and decode_from_latent of 3x40x48x40 latents (BASELINE cfg4 shapes),
    `--batch` volumes per call.  Prints volumes/s for the decode (the step after sampling)."""
    import torch
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.require_device()
    B, K, W = args.batch, args.steps, max(3, args.warmup)
    torch.manual_seed(0)
    vae = VAE3D(4, 32, 3, 3).to(dev).eval()
    x = torch.randn(B, 4, 160, 192, 160, device=dev)
    z = torch.randn(B, *LATENT, device=dev)
    res = {}
    with torch.no_grad():
        for name, fn, inp in (("decode", vae.decode_from_latent, z), ("encode", vae.encode_to_latent, x)):
            for _ in range(W):
                fn(inp)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                out = fn(inp)
            e1.record()
            torch.cuda.synchronize(dev)
            prog = vae._program(name, inp)
            res[name] = {"ms": e0.elapsed_time(e1) / K, "executed_gemm_tflop": prog.gemm_flops / 1e12,
                         "finite": bool(torch.isfinite(out).all().item())}
    # ---- stage 1 of ddpm_3d_ldm/train.py:258-300: one VAE training step at the script's patch size
    # (4 x 128 x 160 x 160, batch 1, VAE3D(4, 32, 3, latent 16)): vae(x) + L1 + KL + backward
    import torch.nn.functional as F

    def vae_loss(recon, xx, mu, logvar):
        kl = -0.5 * torch.mean(1 + logvar - mu.pow(2) - logvar.exp())
        return F.l1_loss(recon, xx) + 1e-4 * kl

    torch.manual_seed(0)
    tv = VAE3D(4, 32, 3, 16).to(dev).train()
    xt = torch.randn(1, 4, 128, 160, 160, device=dev).clamp_(-1, 1)

    def ours_step():
        tv.zero_grad(set_to_none=True)
        recon, mu, logvar = tv(xt)
        vae_loss(recon, xt, mu, logvar).backward()

    def timed(fn, warm, iters):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / iters

    train = {"ms": timed(ours_step, 4, K), "batch": 1, "patch": [128, 160, 160],
             "model": "VAE3D(4, base 32, num_down 3, latent 16) (train.py:43-46)"}
    progs = [p_ for k_, p_ in tv._programs().items() if k_[-1]]
    train["executed_gemm_tflop"] = sum(p_.gemm_flops + p_.bwd_flops for p_ in progs) / 1e12
    train["finite_grads"] = all(bool(torch.isfinite(p_.grad).all().item()) for p_ in tv.parameters())
    if rank == 0 and not args.no_gpu_comparator:
        # the reference's graph (oracle restatement = the same ATen / cuDNN calls) eagerly, autocast bf16
        from oracle import reference_oracle as O
        torch.backends.cudnn.benchmark = True
        sd = {k: v.detach().clone().requires_grad_(True) for k, v in tv.state_dict().items()}

        def eager_step():
            for v in sd.values():
                v.grad = None
            with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
                mu, logvar = O.vae3d_encode(sd, xt)
                zz = mu + torch.randn_like(mu) * torch.exp(0.5 * logvar)
                recon = O.vae3d_decode(sd, zz)
                loss = vae_loss(recon.float(), xt, mu.float(), logvar.float())
            loss.backward()

        train["eager_cudnn_autocast_bf16_ms"] = timed(eager_step, 2, max(2, K // 3))
        del sd
    del tv
    torch.cuda.empty_cache()
    if rank != 0:
        return
    peaks = load_peaks()
    for r in list(res.values()) + [train]:
        r["tflops_executed"] = r["executed_gemm_tflop"] / (r["ms"] * 1e-3)
    line = {"metric": "volumes/sec (VAE3D decode_from_latent, 3x40x48x40 -> 4x160x192x160)",
            "value": world * B / (res["decode"]["ms"] / 1e3), "unit": "volumes/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": res["decode"]["ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "vae3d_decode", "batch_per_gpu": B,
                       "model": "VAE3D(4, base 32, num_down 3, latent 3)",
                       "note": "executed FLOPs include the zero padding of 32-channel layers to 64"},
            "decode": res["decode"], "encode": res["encode"], "train_step": train,
            "peak_tflops": peaks["tflops"]}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=0,
                    help="volumes per GPU (default: 16 for sampling -- measured sweep in "
                         "profiles/README.md: 2 -> 0.59, 4 -> 0.67, 8 -> 0.74, 16 -> 0.76 volumes/s --, "
                         "8 for the training step (BASELINE cfg5), 1 for the VAE)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="sample", choices=["sample", "train", "vae"],
                    help="sample = headline (cfg4); train = DDP training step (cfg5); vae = VAE3D "
                         "encode / decode at the cfg4 volume size")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-comparator", action="store_true",
                    help="skip the eager cuDNN run of the reference graph on the same GPU (N = 1 only)")
    ap.add_argument("--no-train", action="store_true",
                    help="sample mode: skip the cfg5 DDP training-step record appended to the line")
    ap.add_argument("--train-batch", type=int, default=8, help="latents per GPU of the training record")
    ap.add_argument("--train-steps", type=int, default=20, help="timed steps of the training record (<= --steps)")
    ap.add_argument("--torch-adam", action="store_true", help="train mode: torch.optim.Adam instead of "
                    "mri_image_generation_b200.optim.Adam")
    ap.add_argument("--no-ddp", action="store_true", help="train mode, N > 1: independent replicas without "
                    "gradient exchange (attribution of the multi-GPU step time)")
    ap.add_argument("--torch-ddp", action="store_true", help="train mode, N > 1: torch DDP instead of the "
                    "overlapped bucketed all-reduce (parallel.DistributedDataParallel)")
    ap.add_argument("--per-op", default="", help="write per-GEMM timings (CUDA events) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="sample mode: after the timed steps write rank 0's x_{t-1} of the last timed "
                         "step as DIR/x_prev.npy (float32, [batch, 3, 40, 48, 40]; inputs are seeded, "
                         "so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "sample" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the sampling workload (--mode sample --impl ours)")

    if args.batch <= 0:
        args.batch = {"sample": 16, "train": 8, "vae": 1}[args.mode]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.mode == "train":
            run_train(args, rank, world, local_rank)
        elif args.mode == "vae":
            run_vae(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
