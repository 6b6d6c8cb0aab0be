"""Where the device time of one bench.py encoder step goes between kernels.

At the bench shape (4096 segments x 4096 points, bf16 tier, max / mean pooling) it warms up, records --trace-steps steps
under torch.profiler (CUDA activity only) and, in the same process with the profiler off, times --timed-steps steps with
device events.  It writes <out-dir>/<tag>_step_trace.json with every kernel's and memset's start and end, the idle time
before each of them grouped by boundary type (memset->chain, chain->fusion, fusion->chain, step->step = last fusion ->
next memset), the sum of kernel time, the device-timed step, and the card's name, power limit and SM clock (read-only
nvidia-smi queries, sampled through both windows).  A negative idle time is an overlap: the next kernel started before
the previous one ended (programmatic dependent launch).

    python tools/step_trace.py --tag r03a [--segments 4096 --points 4096 --warmup 3 --trace-steps 3 --timed-steps 10]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, sm, smax = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit_w": float(pl), "sm_mhz_idle": float(sm), "sm_max_mhz": float(smax)}
    except Exception as e:  # no nvidia-smi: say so rather than guess
        return {"name": None, "error": repr(e)}


def kind_of(ev):
    name = ev["name"]
    if ev.get("cat") == "gpu_memset" or name.startswith("Memset"):
        return "memset"
    if "chain_pair_kernel" in name:
        return "chain"
    if "gemm_pair_kernel" in name:
        return "fusion"
    return "other"


def analyse(events, steps):
    """events: device events (kind, name, start_us, end_us) sorted by start.  Boundaries are labelled by the kinds of the
    event before and after; step->step is the idle time between a step's last kernel and the next step's memset."""
    groups = {}
    rows = []
    prev = None
    for kind, name, t0, t1 in events:
        row = {"kind": kind, "name": name, "start_us": t0, "end_us": t1, "dur_us": t1 - t0}
        if prev is not None:
            label = "step->step" if kind == "memset" else f"{prev[0]}->{kind}"
            idle = t0 - prev[3]
            row["idle_before_us"] = idle
            g = groups.setdefault(label, [])
            g.append(idle)
        rows.append(row)
        prev = (kind, name, t0, t1)
    first, last = events[0][2], max(e[3] for e in events)
    busy, cur_end = 0.0, None   # union of the kernels' intervals (they may overlap)
    for _, _, t0, t1 in events:
        if cur_end is None or t0 > cur_end:
            busy += t1 - t0
            cur_end = t1
        elif t1 > cur_end:
            busy += t1 - cur_end
            cur_end = t1
    summary = {
        label: {"count": len(v), "sum_us": sum(v), "mean_us": sum(v) / len(v), "min_us": min(v), "max_us": max(v)}
        for label, v in sorted(groups.items())
    }
    kernel_sum = sum(e[3] - e[2] for e in events)
    idle_sum = sum(v for g in groups.values() for v in g if v > 0)
    return rows, {
        "boundaries": summary,
        "traced_span_ms": (last - first) * 1e-3,
        "traced_ms_per_step": (last - first) * 1e-3 / steps,
        "kernel_sum_ms_per_step": kernel_sum * 1e-3 / steps,
        "busy_union_ms_per_step": busy * 1e-3 / steps,
        "idle_ms_per_step": idle_sum * 1e-3 / steps,
        "by_kind_ms_per_step": {k: sum(e[3] - e[2] for e in events if e[0] == k) * 1e-3 / steps
                                for k in sorted({e[0] for e in events})},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--tag", required=True)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--segments", type=int, default=4096)
    ap.add_argument("--points", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--trace-steps", type=int, default=3)
    ap.add_argument("--timed-steps", type=int, default=10)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import pointnet_refine_b200 as prb
    from bench import ClockSampler

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    enc = prb.LineRefineNet().to(dev).eval().context_encoder
    enc.precision = "bf16"
    gen = torch.Generator(device=dev).manual_seed(1234)
    ctx = torch.randn(args.segments, args.points, 4, device=dev, generator=gen)

    def step():
        return enc.run_native(ctx, pool=True)["global_feat"]

    card = card_info()
    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()

        sampler = ClockSampler(0)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.timed_steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        timed_clocks = sampler.stop()
        ms_per_step = e0.elapsed_time(e1) / args.timed_steps

        sampler = ClockSampler(0)
        sampler.start()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.trace_steps):
                step()
            torch.cuda.synchronize()
        traced_clocks = sampler.stop()

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    events = []
    for ev in trace.get("traceEvents", []):
        if ev.get("ph") != "X" or ev.get("cat") not in ("kernel", "gpu_memset"):
            continue
        events.append((kind_of(ev), ev["name"], float(ev["ts"]), float(ev["ts"]) + float(ev["dur"])))
    events.sort(key=lambda e: e[2])
    if not events or events[0][0] != "memset":
        raise SystemExit(f"unexpected trace: first device event {events[0] if events else None}")
    rows, summary = analyse(events, args.trace_steps)
    result = {
        "tag": args.tag,
        "shape": {"segments": args.segments, "points": args.points, "precision": "bf16", "outputs": "pool"},
        "card": card,
        "timed": {"steps": args.timed_steps, "ms_per_step": ms_per_step, "clocks": timed_clocks},
        "traced": {"steps": args.trace_steps, "clocks": traced_clocks, **summary},
        "step_minus_kernels_ms": ms_per_step - summary["kernel_sum_ms_per_step"],
        "step_minus_busy_ms": ms_per_step - summary["busy_union_ms_per_step"],
        "kernels": rows,
    }
    os.makedirs(args.out_dir, exist_ok=True)
    out = os.path.join(args.out_dir, f"{args.tag}_step_trace.json")
    with open(out, "w") as f:
        json.dump(result, f, indent=1)
    brief = {k: v for k, v in result.items() if k != "kernels"}
    print(json.dumps(brief, indent=1))
    print("wrote", out)


if __name__ == "__main__":
    main()
