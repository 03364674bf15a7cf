#!/usr/bin/env python
"""bench.py -- audio-seconds/sec of the VSampler on the README U-Net (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2|cfg3|cfg5] [--impl reference]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one complete `model.sample(...)` call on each rank (weak scaling: the per-GPU batch is
fixed, independent sampling, no collective on the data path).  Prints ONE JSON line (rank 0).
K sets the timed steps of both sampling legs (device, e2e); the training leg is a separate
measurement of a fixed 5 timed steps.

--dump-outputs DIR writes rank 0's result of the last timed device step as DIR/sample.npy (float32,
the whole [batch, 2, 2**18] clip: 16.8 MB for cfg2/cfg5, 33.6 MB for cfg3) and, when the training
leg runs, the loss of its last timed step as DIR/train_loss.npy (float64).  Weights and inputs come
from fixed seeds, so two builds run with the same arguments can be compared output for output.

  --config cfg2 (default, BASELINE configs[1], the configuration `metric` is quoted on):
        unconditional README UNetV0, noise [8,2,2^18] per GPU, 50-step VSampler
  --config cfg3 (configs[2]): text-conditional net (cross-attention at L3..L8, embedding
        [16,64,768]), classifier-free guidance 5.0, batch 16 per GPU, 50 steps
  --config cfg5 (configs[4]): DiffusionVocoder (mel 80 x 1024, n_fft 1024), 8 stereo clips per
        GPU (= 64 over 8 GPUs = 16 mono sequences per GPU), 100 steps

  value     clips*5.4613 s / wall, inputs resident in HBM, device-timed, max over ranks
  e2e       same through the public API from pinned HOST inputs to a HOST result
  roofline  the dominant kernel/shape of the step, timed live with CUDA events in an instrumented
            eager pass of the same plan; `traffic` = DRAM bytes per launch read from the committed
            ncu capture named in `traffic_source` (null when that shape has no capture)
  cpu_baseline  the reference's eager-PyTorch CPU path (oracle port) on this box's host cores,
            bounded sample, extrapolated (stated in `sample`)

`--impl reference` times only that CPU path (rank 0), same metric/config: each of the K timed
steps is ONE VSampler step of the config's batch on clips cut to the longest power-of-two length
for which warmup + K steps fit the time budget; `value` extrapolates to the full workload.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLE_RATE = 48000
LENGTH = 2 ** 18
CLIP_SECONDS = LENGTH / SAMPLE_RATE          # 5.4613 s, stereo counts once
README = dict(in_channels=2, channels=[8, 32, 64, 128, 256, 512, 512, 1024, 1024],
              factors=[1, 4, 4, 4, 2, 2, 2, 2, 2], items=[1, 2, 2, 2, 2, 2, 2, 4, 4],
              attentions=[0, 0, 0, 0, 0, 1, 1, 1, 1], attention_heads=8, attention_features=64)
CFG3 = dict(README, cross_attentions=[0, 0, 0, 1, 1, 1, 1, 1, 1], use_embedding_cfg=True,
            embedding_max_length=64, embedding_features=768)
UNET9 = dict(channels=[8, 32, 64, 128, 256, 512, 512, 1024, 1024],
             factors=[1, 4, 4, 4, 2, 2, 2, 2, 2], items=[1, 2, 2, 2, 2, 2, 2, 4, 4])
VOCODER = dict(mel_n_fft=1024, mel_channels=80, mel_sample_rate=48000, mel_normalize_log=True, **UNET9)
UPSAMPLER = dict(upsample_factor=16, in_channels=2, **UNET9)
METRIC = "audio-seconds/sec (2ch, 2^18 len) VSampler 50-step"
L2_NOTE = ("no explicit flush: one net evaluation streams ~0.9 GB (activations + 435 MB weights), "
           "far beyond the 126 MB L2")

WORKLOADS = {
    "cfg2": dict(batch=8, steps=50, metric=METRIC,
                 workload="configs[1]: unconditional README UNetV0 9-stage, noise randn[8,2,2**18] per "
                          "GPU, VSampler num_steps=50"),
    "cfg3": dict(batch=16, steps=50, metric="audio-seconds/sec (2ch, 2^18 len) VSampler 50-step, text+CFG",
                 workload="configs[2]: text-conditional README UNetV0 (cross_attentions=[0,0,0,1,1,1,1,1,1], "
                          "precomputed embedding randn[16,64,768], CFG scale 5.0), noise randn[16,2,2**18] "
                          "per GPU, VSampler num_steps=50"),
    "cfg5": dict(batch=8, steps=100, metric="audio-seconds/sec (2ch, 2^18 len) DiffusionVocoder 100-step",
                 workload="configs[4]: DiffusionVocoder mel_channels=80 n_fft=1024, mel randn[8,2,80,1024] per "
                          "GPU (64 clips over 8 GPUs = 16 mono sequences per GPU), VSampler num_steps=100"),
}


def workload_config(name: str):
    w = WORKLOADS[name]
    return {"workload": w["workload"], "batch_per_gpu": w["batch"], "length": LENGTH,
            "num_steps": w["steps"], "sample_rate": SAMPLE_RATE, "l2": L2_NOTE}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return p["hbm_gbs"], p["bf16_tflops"], p["bf16_tflops_sustained"], "measured"
    except Exception:
        return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ reference arm
def _host_threads() -> int:
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                      # cgroup v2 CPU quota ("max 100000" = unlimited)
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            avail = max(1, min(avail, int(int(quota) / int(period))))
    except Exception:
        pass
    return avail


def cpu_reference_run(config: str, steps: int, warmup: int, budget_s: float, batch=None):
    """The reference's own eager CPU path (oracle port over the a_unet shim), fp32, host threads.
    One timed unit = ONE VSampler step (reference diffusion.py:183-188: every step costs the same)
    of the config's per-GPU batch, on clips of the largest power-of-two length <= 2**18 for which
    warmup + steps units fit `budget_s` (probed at 2**13).  value = audio-seconds/sec of the full
    num_steps sampler extrapolated from that unit.  Shorter clips are slightly CHEAPER per audio
    second (attention is quadratic in length), so a bounded sample can only flatter the CPU arm.
    Returns (value, seconds per unit, threads, description)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_port as port
    w = WORKLOADS[config]
    batch = w["batch"] if batch is None else batch
    torch.manual_seed(0)
    if config == "cfg5":
        model = port.DiffusionVocoderPort(**VOCODER)
    else:
        model = port.DiffusionModelPort(**(CFG3 if config == "cfg3" else README))

    def one_step(length):
        if config == "cfg5":
            mel = torch.randn(batch, 2, 80, length // 256)
            t0 = time.perf_counter()
            with torch.no_grad():
                model.sample(mel, num_steps=1)
        else:
            x = torch.randn(batch, 2, length)
            kw = dict(embedding=torch.randn(batch, 64, 768), embedding_scale=5.0) if config == "cfg3" else {}
            t0 = time.perf_counter()
            with torch.no_grad():
                model.sample(x, num_steps=1, **kw)
        return time.perf_counter() - t0

    # "all the host threads it can use": the count that actually runs this path fastest.  On a
    # box whose cgroup grants fewer CPUs than os.cpu_count() reports, cpu_count() threads
    # time-slice and every OpenMP barrier stalls (measured: 47 s per unit at 128 threads), so
    # the thread count is probed upwards from 8 on a short clip and the best one kept.
    avail = _host_threads()
    probe_len = 2 ** 13
    cores, t_probe = None, None
    for n in [c for c in (8, 16, 32, 64, 128, 256) if c < avail] + [avail]:
        torch.set_num_threads(n)
        one_step(2 ** 12)                     # thread pool / allocator warm at this width
        t = one_step(probe_len)
        if t_probe is not None and t > 0.9 * t_probe:
            if t < t_probe:
                cores, t_probe = n, t
            break                             # no longer scaling
        cores, t_probe = n, t
    torch.set_num_threads(cores)
    length = probe_len
    units = max(steps + warmup, 1)
    while length < LENGTH and units * t_probe * (2 * length / probe_len) <= budget_s:
        length *= 2
    times = []
    for i in range(warmup + steps):
        dt = one_step(length)
        if i >= warmup:
            times.append(dt)
    per_step = sum(times) / len(times)
    value = batch * CLIP_SECONDS * (length / LENGTH) / (w["steps"] * per_step)
    return value, per_step, cores, (
        f"{len(times)} timed x ONE VSampler step on batch {batch} of [2,{length}] fp32 ({cores} threads; "
        f"the full clip is 2**18 = {LENGTH} samples), value = batch*clip_seconds*(length/2**18) / "
        f"({w['steps']} steps x measured seconds per step)")


def run_reference(args, rank: int):
    if rank != 0:
        return
    w = WORKLOADS[args.config]
    value, per_step, cores, sample = cpu_reference_run(args.config, args.steps, args.warmup, budget_s=200.0)
    line = {"impl": "reference", "metric": w["metric"], "value": value, "unit": "audio-s/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_step * 1e3,        # measured: one timed unit (see cpu_baseline.sample)
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.config),
            "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    emit(json.dumps(line))


# ------------------------------------------------------------------------------- training leg
def train_step_bench(adp, dev, world, dist, steps, warmup, batch=4):
    """BASELINE configs[3]: DiffusionUpsampler(upsample_factor=16) training step -- fused loss,
    hand-written backward, gradient all-reduce over NCCL when world > 1, fused AdamW --
    `batch` clips of [2, 2**18] per GPU.  Returns ms per step (device-timed, max over ranks)."""
    from audio_diffusion_pytorch_b200 import parallel
    model = adp.DiffusionUpsampler(net_t=adp.UNetV0, **UPSAMPLER).to(dev)
    step_model = model
    if world > 1:
        step_model = parallel.OverlappedDataParallel(model)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True)
    audio = torch.randn(batch, 2, LENGTH, device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = step_model(audio)
        loss.backward()
        if world > 1:
            step_model.finish_gradient_sync()
        opt.step()
        return loss

    for _ in range(max(warmup, 3)):
        step()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return {"ms_per_step": float(ms.item()), "loss": float(loss.detach()), "batch_per_gpu": batch,
            "config": "configs[3]: DiffusionUpsampler upsample_factor=16, [B,2,2**18], fwd+bwd+"
                      "AdamW" + ("+NCCL grad all-reduce overlapped with the backward program" if world > 1 else ""),
            "audio_s_per_s": batch * world * CLIP_SECONDS / (float(ms.item()) * 1e-3)}


# --------------------------------------------------------------------------- ncu-derived traffic
def ncu_traffic(kernel_label: str):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full`
    capture) for a kernel/shape label, from profiles/ncu_traffic.json -- written by
    tools/ncu_traffic.py from the committed captures.  (None, None) when that shape has none."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            table = json.load(fh)
        ent = table.get(kernel_label)
        if ent:
            return float(ent["dram_bytes"]), ent["source"]
    except Exception:
        pass
    return None, None


# stdout carries exactly ONE JSON line: libraries that print to fd 1 from C (NCCL's version
# banner) are sent to stderr for the duration of the run
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(text: str):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (text + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-ops", action="store_true", help="print the per-kernel table")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import audio_diffusion_pytorch_b200 as adp
    torch.manual_seed(1234 + rank)
    w = WORKLOADS[args.config]
    batch, num_steps = w["batch"], w["steps"]
    warmup = max(args.warmup, 3)
    host_kw, kw = {}, {}
    if args.config == "cfg5":
        model = adp.DiffusionVocoder(net_t=adp.UNetV0, **VOCODER).to(dev)
        host_in = torch.randn(batch, 2, 80, LENGTH // 256).pin_memory()      # mel spectrogram
    else:
        model = adp.DiffusionModel(net_t=adp.UNetV0, **(CFG3 if args.config == "cfg3" else README)).to(dev)
        host_in = torch.randn(batch, 2, LENGTH).pin_memory()                 # starting noise
        if args.config == "cfg3":
            host_kw = {"embedding": torch.randn(batch, 64, 768).pin_memory()}
            kw = {"embedding_scale": 5.0}
    net = model.net
    host_out = torch.empty(batch, 2, LENGTH).pin_memory()
    dev_in = host_in.to(dev)
    dev_kw = {k: v.to(dev) for k, v in host_kw.items()}

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, iters):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    outputs = {}

    def step_device():
        outputs["sample"] = model.sample(dev_in, num_steps=num_steps, **dev_kw, **kw)

    def step_e2e():
        x = host_in.to(dev, non_blocking=True)
        k2 = {k: v.to(dev, non_blocking=True) for k, v in host_kw.items()}
        out = model.sample(x, num_steps=num_steps, **k2, **kw)
        host_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(warmup):
        step_device()
    with ClockSampler(local) as clocks:
        total_ms = timed(step_device, args.steps)
    last_sample = outputs.pop("sample")
    dumps = {"sample": last_sample.float().cpu().numpy()} if args.dump_outputs else {}
    del last_sample
    for _ in range(2):
        step_e2e()
    e2e_ms = timed(step_e2e, args.steps)

    ms_per_step = total_ms / args.steps
    clips = batch * world
    value = clips * CLIP_SECONDS / (ms_per_step * 1e-3)
    e2e_value = clips * CLIP_SECONDS / (e2e_ms / args.steps * 1e-3)

    roof, table = None, {}
    plan = next(p for k, p in net._plans.items() if len(k) > 4 and k[4] == "sample")
    cond_plan = next((p for k, p in net._plans.items() if k[0] == "cond"), None)
    n_kernels, n_pre = plan.n_kernels, len(getattr(plan, "pre", []))
    if rank == 0:      # profiling passes (no collectives inside): rank 0 only
        # ---- roofline of the dominant kernel/shape of one net evaluation.
        # (1) in-graph durations per kernel + shape: the step's CUDA graph re-captured with programmatic
        #     dependent launch OFF (with PDL a kernel's duration includes the time it waits for its
        #     predecessor) and replayed under CUPTI activity tracing, AFTER the timed region;
        # (2) the same launches timed with CUDA events in an eager pass of the plan (upper bound:
        #     includes host launch gaps).  `achieved` uses (1); (2) is reported next to it.
        from audio_diffusion_pytorch_b200 import _lib
        table = net.profile_plan(plan, iters=5)
        hbm, tf_burst, tf_sust, which = peaks()
        gtab, busy_us, in_graph_err = None, None, None
        try:
            from tools.graph_profile import in_graph_table
            saved = dict(net._plans)
            net._plans.clear()
            _lib.lib().adp_debug_set(6, 0)
            try:
                for _ in range(2):
                    model.sample(dev_in, num_steps=2, **dev_kw, **kw)
                plan_np = next(p for k, p in net._plans.items() if len(k) > 4 and k[4] == "sample")
                gtab, _, busy_us, _ = in_graph_table(
                    net, plan_np, lambda k: model.sample(dev_in, num_steps=k, **dev_kw, **kw), 4)
            finally:
                _lib.lib().adp_debug_set(6, 1)
                net._plans.clear()
                net._plans.update(saved)
        except Exception as exc:                      # profiler unavailable: event-timed numbers only
            in_graph_err = repr(exc)[:200]
        if gtab:
            top_name = max(gtab, key=lambda k: gtab[k]["us_total"])
            top_us, top_share = gtab[top_name]["us_avg"], gtab[top_name]["us_total"] / busy_us
            top = table.get(top_name) or {"name": top_name, "flops": gtab[top_name]["flops"],
                                          "bytes": gtab[top_name]["bytes"], "count": gtab[top_name]["count"],
                                          "ms_avg": float("nan"), "ms_total": float("nan")}
        else:
            top = max(table.values(), key=lambda r: r["ms_total"])
            top_us = top["ms_avg"] * 1e3
            top_share = top["ms_total"] / sum(r["ms_total"] for r in table.values())
        ai = top["flops"] / max(top["bytes"], 1)
        tensor_bound = ai >= tf_sust * 1e12 / (hbm * 1e9)
        work, peak, unit = ((top["flops"] / 1e6, tf_sust, "TFLOP/s") if tensor_bound
                            else (top["bytes"] / 1e3, hbm, "GB/s"))
        achieved = work / top_us
        roof = {"bound": "tensor" if tensor_bound else "hbm", "achieved": achieved, "peak": peak, "unit": unit,
                "frac": achieved / peak, "kernel_us": top_us,
                "timing": ("in-graph (CUDA graph of the step re-captured with PDL off, CUPTI activity records, "
                           "4 steps averaged)" if gtab else "CUDA events around each launch of an eager pass"),
                "achieved_eager_events": work / (top["ms_avg"] * 1e3), "eager_event_us": top["ms_avg"] * 1e3}
        if in_graph_err:
            roof["in_graph_error"] = in_graph_err
        if busy_us is not None:
            roof["kernel_busy_us_per_net_eval"] = busy_us
        traffic, traffic_src = ncu_traffic(top["name"])
        roof.update({"kernel": top["name"], "launches_per_net_eval": top["count"],
                     "share_of_step": top_share, "peak_source": which,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "flops_per_launch": top["flops"], "bytes_per_launch": top["bytes"]})
        # whole-step roofline (SURVEY.md 8d): sum over levels of max(flop time, byte time)
        t_bound = sum(max(r["flops"] / (tf_sust * 1e12), r["bytes"] / (hbm * 1e9)) * r["count"]
                      for r in table.values())
        roof["step_bound_ms"] = t_bound * 1e3
        roof["step_frac"] = t_bound * 1e3 / (ms_per_step / num_steps)
    if args.profile_ops and rank == 0:
        for r in sorted(table.values(), key=lambda r: -r["ms_total"]):
            print(f"# {r['name']:58s} x{r['count']:3d} avg {r['ms_avg'] * 1e3:8.1f} us  "
                  f"total {r['ms_total'] * 1e3:9.1f} us  {r['flops'] / max(r['ms_avg'], 1e-9) / 1e9:8.1f} TF/s "
                  f"{r['bytes'] / max(r['ms_avg'], 1e-9) / 1e6:8.1f} GB/s", file=sys.stderr)

    h2d = host_in.numel() * 4 + sum(v.numel() * 4 for v in host_kw.values())
    line = {"metric": w["metric"], "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": dict(workload_config(args.config), parallelism=f"dp{world} (independent sampling)"),
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": host_out.numel() * 4},
            # per step the net's kernels; per sample() call the conditioning (+ context K/V) launches
            "gpu_launches": (n_kernels * num_steps + (6 if cond_plan is not None else 0) + n_pre) * args.steps,
            "ms_per_net_eval": ms_per_step / num_steps,
            "roofline": roof}
    if not args.no_train and args.config == "cfg2":
        del model, net, plan
        gtab = table = None
        torch.cuda.empty_cache()
        line["train_step"] = train_step_bench(adp, dev, world, dist, steps=5, warmup=3)
        dumps["train_loss"] = np.float64(line["train_step"]["loss"])
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        v, per_step, cores, sample = cpu_reference_run(args.config, steps=1, warmup=1, budget_s=25.0, batch=1)
        line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port",
                                "sample": sample}
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumps.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    if rank == 0:
        emit(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
