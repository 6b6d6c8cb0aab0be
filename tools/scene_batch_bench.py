"""Training batches from many device-resident scenes: batches/s of SceneTrainingSet (one lrn_scenes_segments call per
batch) against one K = 1 call per scene (build_training_batch) over the same samples, the host formulation per item
(oracle/scene_oracle.build_segment, a few items), and the time of a replayed GraphedTrainStep at the same shape.
Synthetic scenes (scene_oracle.synth_scene).  Prints one JSON line with the card's name, power limit and the SM clock /
board power sampled while the batches are built.

    python tools/scene_batch_bench.py [--scenes 40] [--points 2000000] [--batch 1024] [--N 2048] [--radius 4.0]
                                      [--batches 5] [--oracle-items 2] [--no-train-step]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import pointnet_refine_b200 as prb  # noqa: E402
from oracle import scene_oracle as so  # noqa: E402
from pointnet_refine_b200 import data  # noqa: E402
from pointnet_refine_b200 import scene as sc  # noqa: E402


def smi(fields):
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True).stdout.strip()
    return [v.strip() for v in out.split(",")] if out else None


class Sampler:
    """SM clock and board power every 100 ms while a timed loop runs."""
    def __init__(self):
        self.samples, self._stop = [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            v = smi("clocks.sm,power.draw")
            if v:
                self.samples.append((float(v[0]), float(v[1])))
            self._stop.wait(0.1)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join()

    def summary(self):
        if not self.samples:
            return None
        c, p = sorted(s[0] for s in self.samples), sorted(s[1] for s in self.samples)
        return {"sm_clock_mhz_median": c[len(c) // 2], "power_w_median": p[len(p) // 2], "samples": len(c)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=40)
    ap.add_argument("--points", type=int, default=2_000_000)
    ap.add_argument("--extent", type=float, default=120.0)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--N", type=int, default=2048)
    ap.add_argument("--radius", type=float, default=4.0)
    ap.add_argument("--batches", type=int, default=5)
    ap.add_argument("--oracle-items", type=int, default=2)
    ap.add_argument("--no-train-step", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scene_batch_bench.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda:0")
    name, power_limit, max_clock = smi("name,power.limit,clocks.max.sm") or (None, None, None)
    lines_per_scene = -(-a.batch // a.scenes) + 2
    scenes, samples = [], []
    rs = np.random.default_rng(0)
    for k in range(a.scenes):
        pts, lines = so.synth_scene(a.points, lines_per_scene, seed=1000 + k, extent=a.extent)
        scenes.append(pts)
        samples += [(k, raw, raw + rs.normal(0, 0.2, raw.shape)) for raw in lines]
    t0 = time.perf_counter()
    prepared = sc.prepare_scenes([torch.from_numpy(p).to(dev) for p in scenes])
    torch.cuda.synchronize()
    t_prepare = time.perf_counter() - t0
    t0 = time.perf_counter()
    ts = data.SceneTrainingSet(prepared, samples, a.batch, a.N, a.radius, 2.0, seed=0)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    order = ts.order()
    batches = [order[(b * a.batch) % (len(samples) - a.batch + 1):][:a.batch] for b in range(a.batches + 1)]

    # (a) SceneTrainingSet: one call per batch
    ts.batch(batches[0])                                  # warm-up: modules, allocator, capacity
    torch.cuda.synchronize()
    launches = prb._lib.launch_counter
    with Sampler() as clk:
        t0 = time.perf_counter()
        for b in batches[1:]:
            ts.batch(b)
        torch.cuda.synchronize()
        t_set = (time.perf_counter() - t0) / a.batches
    launches = (prb._lib.launch_counter - launches) / a.batches

    # (b) one K = 1 call per scene (build_training_batch) over the same samples
    def per_scene(idx):
        idx = idx.cpu().numpy()
        for k in np.unique([samples[i][0] for i in idx]):
            own = [i for i in idx if samples[i][0] == k]
            sc.build_training_batch(prepared.scene(int(k)), [samples[i][1] for i in own], [samples[i][2] for i in own],
                                    a.N, a.radius, 2.0, seed=0)
    per_scene(batches[0])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in batches[1:]:
        per_scene(b)
    torch.cuda.synchronize()
    t_loop = (time.perf_counter() - t0) / a.batches
    scenes_per_batch = float(np.mean([len({samples[i][0] for i in b.tolist()}) for b in batches[1:]]))

    # (c) the host formulation per item
    t_item = None
    if a.oracle_items > 0:
        t0 = time.perf_counter()
        for i in range(a.oracle_items):
            k, raw, _ = samples[i]
            so.build_segment(scenes[k], raw, a.N, a.radius, 2.0, 0, i)
        t_item = (time.perf_counter() - t0) / a.oracle_items

    # replayed train step at the batch's shape
    t_step = None
    if not a.no_train_step:
        from pointnet_refine_b200.optim import FlatAdam
        torch.manual_seed(0)
        m = prb.LineRefineNet().to(dev).train()
        m.context_encoder.native_training = True
        batch = ts.batch(batches[0])
        step = prb.GraphedTrainStep(m, FlatAdam(m.parameters(), lr=1e-4, capturable=True), batch["context"],
                                    batch["noisy_line"], batch["target_offset"])
        step(batch["context"], batch["noisy_line"], batch["target_offset"])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            step(batch["context"], batch["noisy_line"], batch["target_offset"])
        torch.cuda.synchronize()
        t_step = (time.perf_counter() - t0) / 5

    print(json.dumps({
        "gpu": name, "power_limit_w": power_limit, "max_sm_clock_mhz": max_clock, "during_scene_training_set": clk.summary(),
        "scenes": a.scenes, "points_per_scene": a.points, "extent_m": a.extent, "samples": len(samples), "batch": a.batch,
        "N": a.N, "crop_radius": a.radius, "scenes_per_batch": scenes_per_batch,
        "prepare_scenes_s": round(t_prepare, 3), "training_set_setup_s": round(t_setup, 3),
        "scene_training_set": {"ms_per_batch": round(t_set * 1e3, 2), "batches_per_s": round(1 / t_set, 2),
                               "samples_per_s": round(a.batch / t_set, 1), "library_launches_per_batch": launches},
        "one_k1_call_per_scene": {"ms_per_batch": round(t_loop * 1e3, 2), "batches_per_s": round(1 / t_loop, 2)},
        "host_oracle_per_item": None if t_item is None else {"ms_per_item": round(t_item * 1e3, 1),
                                                             "batches_per_s": round(1 / (t_item * a.batch), 5)},
        "graphed_train_step": None if t_step is None else {"ms_per_step": round(t_step * 1e3, 2),
                                                           "batch_build_over_step": round(t_set / t_step, 3)},
    }), flush=True)


if __name__ == "__main__":
    main()
