"""Transfer-learning train step (context encoder frozen: `.eval().requires_grad_(False)`, FlatAdam over the trainable
parameters) against the full native train step, at B x N points and M = 32 polyline points (default 1024 x 1024).

Arms:
  frozen_native : the frozen encoder with the `native_training` opt-in: eval encoder (LRN_OUT_FUSED_BF16) + native train decoder
  full_native   : every parameter trains, `native_training` on: train encoder forward + backward + native train decoder
  frozen_stock  : the frozen encoder without the opt-in (the baseline): eval encoder with fp32 `fused`, stock context_proj
                  and stock fp32 decoder
Each arm's peak memory is measured on its own first (eager steps, then capture), then the arms' eager steps and CUDA-graph
replays (GraphedTrainStep) are timed in alternating rounds, the order reversed every round; every figure is reported as
min / median / max over the rounds.  Prints one JSON line with the card's name, power limit and SM clock limit.
python tools/frozen_train_bench.py [--segments 1024] [--points 1024] [--rounds 3] [--steps 8] [--arms a,b,c]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointnet_refine_b200 as prb  # noqa: E402
from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1  # noqa: E402

ARMS = ("frozen_native", "full_native", "frozen_stock")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class Arm:
    def __init__(self, name, dev, ctx, line, tgt):
        torch.manual_seed(0)
        m = prb.LineRefineNet().to(dev).train()
        if name.startswith("frozen"):
            m.context_encoder.eval().requires_grad_(False)
        m.context_encoder.native_training = name != "frozen_stock"
        self.name, self.dev, self.model = name, dev, m
        self.batch = (ctx, line, tgt)
        self.opt = FlatAdam([p for p in m.parameters() if p.requires_grad], lr=1e-4, capturable=True)
        self.graph = None

    def eager(self):
        ctx, line, tgt = self.batch
        self.opt.zero_grad()
        loss = deep_supervision_l1(self.model(ctx, line), tgt)
        loss.backward()
        self.opt.step()
        return loss.detach()

    def replay(self):
        return self.graph(*self.batch)[0]

    def capture(self):
        self.graph = prb.GraphedTrainStep(self.model, self.opt, *self.batch)


def timed(fn, steps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(out)


def spread(xs):
    xs = sorted(xs)
    return {"min": round(xs[0], 2), "median": round(xs[len(xs) // 2], 2), "max": round(xs[-1], 2), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=1024)
    ap.add_argument("--points", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--arms", default=",".join(ARMS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frozen_train_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    B, N = args.segments, args.points
    g = torch.Generator(device=dev).manual_seed(100)
    ctx = torch.randn(B, N, 4, device=dev, generator=g)
    line = torch.randn(B, 32, 3, device=dev, generator=g)
    tgt = 0.1 * torch.randn(B, 32, 3, device=dev, generator=g)
    names = [a for a in args.arms.split(",") if a]
    res = {"card": card(), "segments": B, "points": N, "M": 32, "steps_per_timing": args.steps, "arms": {}}
    arms = {}
    for name in names:       # peak memory of each arm on its own: eager steps, then the capture
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        arm = arms[name] = Arm(name, dev, ctx, line, tgt)
        for _ in range(2):
            arm.eager()
        torch.cuda.synchronize()
        r = res["arms"][name] = {"peak_mem_gb_eager": (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 30}
        try:
            arm.capture()
            torch.cuda.synchronize()
            r["peak_mem_gb_with_graph"] = (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 30
        except Exception as e:      # report the eager figures and say why
            r["graph_note"] = f"{type(e).__name__}: {e}"[:300]
        r["eager_ms"], r["replay_ms"], r["loss"] = [], [], None
    for rnd in range(args.rounds):
        order = names if rnd % 2 == 0 else names[::-1]
        for name in order:
            arm, r = arms[name], res["arms"][name]
            ms, r["loss"] = timed(arm.eager, args.steps)
            r["eager_ms"].append(ms)
            if arm.graph is not None:
                r["replay_ms"].append(timed(arm.replay, args.steps)[0])
    for name in names:
        r = res["arms"][name]
        r["eager_ms"] = spread(r["eager_ms"])
        r["replay_ms"] = spread(r["replay_ms"]) if r["replay_ms"] else None
        r["peak_mem_gb_eager"] = round(r["peak_mem_gb_eager"], 2)
        if "peak_mem_gb_with_graph" in r:
            r["peak_mem_gb_with_graph"] = round(r["peak_mem_gb_with_graph"], 2)
        if arms[name].graph is not None:
            arms[name].graph.close()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
