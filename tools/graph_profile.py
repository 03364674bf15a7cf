"""In-graph kernel durations PER SHAPE of one sampling step (CUPTI through torch.profiler sees the
kernels of a CUDA-graph replay).  A graph replays the plan's launches in program order, so the
i-th adp kernel of a step is the i-th record of an `ops.trace()` pass over the same plan: that
gives every in-graph duration its label (kernel + M/K/N shape) and algorithmic flops / bytes.

    python tools/graph_profile.py [cfg2|cfg3|cfg5] [steps] [pdl]      -> table on stdout

`in_graph_table()` is also used by bench.py (roofline.achieved_in_graph)."""
import os
import sys
from collections import defaultdict

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def in_graph_table(net, plan, run_steps, steps: int):
    """run_steps(n): runs n sampling steps through the captured graph of `plan`.
    Returns ({label: {count, us_avg, us_total, flops, bytes}} per step, kernels per step,
    kernel-busy us per step, span us per step)."""
    from audio_diffusion_pytorch_b200 import ops
    if hasattr(plan, "step"):
        plan.step.zero_()
    with ops.trace() as tr:
        plan.run_eager()
    torch.cuda.synchronize()
    labels = tr.records
    run_steps(2)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_steps(steps)
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    span = (max(e.time_range.end for e in evs) - min(e.time_range.start for e in evs)) / steps
    ks = sorted((e for e in evs if "adp::" in e.name), key=lambda e: e.time_range.start)
    n = len(labels)
    # the step program's kernels come in runs of n; anything else (conditioning table, context
    # K/V before the loop) precedes the first step
    extra = len(ks) - n * steps
    assert extra >= 0, f"{len(ks)} adp kernels in {steps} steps, expected >= {n} per step"
    ks = ks[extra:]
    table = defaultdict(lambda: {"count": 0, "us_total": 0.0, "flops": 0.0, "bytes": 0.0})
    busy = 0.0
    for i, e in enumerate(ks):
        rec = labels[i % n]
        row = table[rec["name"]]
        us = e.time_range.end - e.time_range.start
        row["count"] += 1
        row["us_total"] += us
        row["flops"], row["bytes"] = rec["flops"], rec["bytes"]
        busy += us
    out = {}
    for name, row in table.items():
        out[name] = {"count": row["count"] / steps, "us_avg": row["us_total"] / row["count"],
                     "us_total": row["us_total"] / steps, "flops": row["flops"], "bytes": row["bytes"]}
    return out, n, busy / steps, span


def format_table(table, n, busy, span, hbm_gbs=6576.4, tflops=1433.0):
    lines = [f"in-graph, per step: {n} kernels, kernel-busy {busy:.1f} us, span {span:.1f} us"]
    lines.append(f"{'kernel / shape':62s} {'x':>5s} {'avg us':>8s} {'us/step':>9s} {'TF/s':>7s} {'GB/s':>7s} "
                 f"{'frac':>5s}")
    for name, r in sorted(table.items(), key=lambda kv: -kv[1]["us_total"]):
        tf = r["flops"] / r["us_avg"] / 1e6
        gb = r["bytes"] / r["us_avg"] / 1e3
        frac = max(tf / tflops, gb / hbm_gbs)
        lines.append(f"{name[:62]:62s} {r['count']:5.0f} {r['us_avg']:8.2f} {r['us_total']:9.1f} {tf:7.1f} "
                     f"{gb:7.1f} {frac:5.2f}")
    return "\n".join(lines)


def main():
    import audio_diffusion_pytorch_b200 as adp
    from audio_diffusion_pytorch_b200 import _lib
    import bench
    cfg = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
    pdl = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    _lib.lib().adp_debug_set(6, pdl)        # programmatic dependent launch on/off (before capture)
    torch.manual_seed(0)
    w = bench.WORKLOADS[cfg]
    kw = {}
    if cfg == "cfg5":
        model = adp.DiffusionVocoder(net_t=adp.UNetV0, **bench.VOCODER).cuda()
        x = torch.randn(w["batch"], 2, 80, 1024, device="cuda")
    else:
        model = adp.DiffusionModel(net_t=adp.UNetV0, **(bench.CFG3 if cfg == "cfg3" else bench.README)).cuda()
        x = torch.randn(w["batch"], 2, 2 ** 18, device="cuda")
        if cfg == "cfg3":
            kw = dict(embedding=torch.randn(w["batch"], 64, 768, device="cuda"), embedding_scale=5.0)
    for _ in range(2):
        model.sample(x, num_steps=3, **kw)          # eager + capture
    plan = next(p for k, p in model.net._plans.items() if len(k) > 4 and k[4] == "sample")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    model.sample(x, num_steps=20, **kw)
    e1.record()
    torch.cuda.synchronize()
    print(f"{cfg} pdl={pdl}: un-profiled {e0.elapsed_time(e1) * 1e3 / 20:.1f} us per step")
    table, n, busy, span = in_graph_table(model.net, plan, lambda k: model.sample(x, num_steps=k, **kw), steps)
    print(format_table(table, n, busy, span))


if __name__ == "__main__":
    main()
