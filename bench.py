#!/usr/bin/env python
"""Benchmark of the LineRefineNet forward hot path (BASELINE.json metric: segments/s & points/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- encoder forward (shared MLP, fusion, gate,
max+mean pooling -> global_feat) over 4096 segments x 4096 context points per GPU, synthetic
N(0,1) points, random-init weights (PyTorch default init, seed 0), bf16 tensor-core tier.  A "step" is one
pass over that batch.  N > 1 (under torchrun): every rank runs the same per-GPU workload on its
own shard, no data-path collective (segments are independent) -> weak scaling.

  value      : whole-job segments/s with the input batch resident in HBM (device-timed, max over ranks)
  e2e        : same metric through the public API from pinned HOST buffers (pointnet_refine_b200.stream.
               HostEncoderPipeline): H2D copy of the context in 512-segment chunks overlapped with the encoder,
               D2H read of global_feat, every step
  roofline   : fusion GEMM kernel (72.7 % of the FLOPs): algorithmic FLOP per launch / mean launch
               duration from CUDA events recorded around each launch (lrn_profile_*), against the
               sustained bf16 peak of MEASURED_PEAKS.json; `chain_kernel` is the same for the fused conv1..conv5 kernel
  --dump-outputs DIR : after the timed steps, DIR/global_feat.npy holds the global_feat (float32) of the last timed step
               on rank 0: (B, 2048), or a fixed sample of its rows (numpy default_rng(0)) when that exceeds 64 MB.  The
               inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
  cpu_baseline / --impl reference : the reference's OWN module (oracle/_ref/src/model.py, staged by oracle/make_ref.py
               from /root/reference in the build container; kind "reference") on the host cores, bounded sample;
               the op-for-op port oracle/torch_port.py (kind "port") only if the staged copy is absent.

Extra keys, measured on rank 0 / all ranks after the timed region (bounded, a few seconds in total):
  full_model     : whole LineRefineNet.forward at the configs[1] shape (4096 x 4096, chunked inside the module)
  config5        : BASELINE configs[4], 256 segments x 65,536 points, encoder + pooling, with property spot checks
  config3_sample : BASELINE configs[2] (1M segments x 2048 points, strong-scaled over the ranks): every rank runs a
                   sample of its shard through the whole forward; seconds for the full 1M sweep extrapolated linearly
  train_step     : BASELINE configs[3], 1024 segments x 1024 points per GPU: forward + L1 deep-supervision loss +
                   backward + Adam on the native train path (FlatDataParallel: flat gradient buffer + NCCL all-reduce when N > 1)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_POINT_ENCODER = 5_587_584      # SURVEY.md section 8d
FLOP_PER_POINT_FUSION_KERNEL = 2 * (1984 + 64) * 1024   # fusion conv + gate layer 2 = 4,194,304
FLOP_PER_POINT_CHAIN_KERNEL = 2 * (64 * 128 + 128 * 256 + 256 * 512 + 512 * 1024)   # conv2..conv5 = 1,392,640
FLOP_PER_POINT_FORWARD = 8_013_952      # whole LineRefineNet.forward per context point (+ 0.399 GFLOP per segment)
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
# SURVEY.md section 8d: 26.4 TFLOP per 1024 x 1024 step / measured peaks (pure-FLOP bound).  "dataflow": the floor of the step as it
# is built (DESIGN.md section 6): every GEMM at the larger of its tensor time and its HBM time (17.4 ms,
# profiles/r02u_train_gemm_shapes.jsonl: seven of the nine layers are HBM-bound at this batch), the BatchNorm / gate passes
# (10.3 ms) and the attention K / V / dK / dV traffic (3.0 ms) at the measured copy bandwidth, ~3 ms of query-side work.
TRAIN_BOUND_MS = {"burst": 16.2, "sustained": 19.3, "dataflow": 34.0}
DUMP_LIMIT_BYTES = 64_000_000


def dump_global_feat(out_dir: str, gf) -> None:
    """Write gf (B, 2048) as out_dir/global_feat.npy; above DUMP_LIMIT_BYTES, a seeded sample of its rows in index order."""
    import numpy as np
    arr = gf.float().cpu().numpy()
    if arr.nbytes > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4096) // arr[0].nbytes         # room for the .npy header
        arr = arr[np.sort(np.random.default_rng(0).choice(len(arr), keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "global_feat.npy"), arr)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return dict(FALLBACK_PEAKS), "fallback"


def tf32_peak(peaks):
    """Sustained cuBLAS tf32 8192^3 figure measured on this pool with the MEASURED_PEAKS.json method
    (tools/cublas_peak.py -> profiles/r02_cublas_peak.json); half the bf16 figure if that file is missing."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_cublas_peak.json")) as f:
            return float(json.load(f)["tf32"]["sustained_tflops"]), "profiles/r02_cublas_peak.json tf32 sustained (cuBLAS 8192^3)"
    except Exception:
        return 0.5 * float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])), "0.5 x bf16_tflops_sustained (no tf32 measurement)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU, sampled every 200 ms while active."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort(); pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": pw[len(pw) // 2] if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------- CPU arm
def _reference_callables():
    """(kind, encoder(ctx_bcn) -> (gf, fused), forward(ctx, line) -> out): the staged reference module if present,
    else the torch-CPU port."""
    import torch
    from oracle import make_ref, synth, torch_port
    sd = synth.to_torch(synth.make_state_dict(0))
    ref = make_ref.load()
    if ref is not None:
        m = ref.LineRefineNet()
        m.load_state_dict(sd, strict=True)
        m.eval()
        return "reference", m.context_encoder, m
    return "port", (lambda x: torch_port.encoder_forward(sd, x)), (lambda c, l: torch_port.line_refine_forward(sd, c, l))


def cpu_reference_run(segments: int, points: int, steps: int, warmup: int, threads: int | None = None, full_forward: bool = False):
    """Time the reference's encoder (or whole forward) on `threads` host threads (default: all) -> segments/s."""
    import torch
    from oracle import synth
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    kind, encoder, forward = _reference_callables()
    ctx_np, line_np = synth.make_inputs(segments, points, seed=1234)
    ctx, line = torch.from_numpy(ctx_np), torch.from_numpy(line_np)
    ctx_t = ctx.transpose(2, 1)
    fn = (lambda: forward(ctx, line)) if full_forward else (lambda: encoder(ctx_t))
    with torch.no_grad():
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        dt = (time.perf_counter() - t0) / steps
    return segments / dt, dt, torch.get_num_threads(), kind


def kind_text(kind):
    return ("the reference's own src/model.py (staged copy, oracle/_ref)" if kind == "reference"
            else "torch-CPU port of the reference (oracle/torch_port.py)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--segments", type=int, default=4096, help="segments per GPU")
    ap.add_argument("--points", type=int, default=4096, help="context points per segment")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32"])
    ap.add_argument("--cpu-sample-segments", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip full_model / config5 / config3_sample / train_step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's global_feat to DIR/global_feat.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")

    # stdout carries exactly ONE line, the result: anything libraries print to fd 1 meanwhile (NCCL's version banner,
    # warnings) goes to stderr
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(result_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    workload = (f"encoder forward + max/mean pooling (global_feat), {args.segments} segments x {args.points} points "
                f"per GPU (BASELINE.json configs[1])")
    config = {"workload": workload, "segments_per_gpu": args.segments, "points_per_segment": args.points,
              "tier": args.precision, "parallelism": f"dp{world} (independent segment shards, no collective)",
              "l2": "input batch (268 MB/GPU at the default size) and per-wave operand buffer (1.24 GB) exceed the 126 MB L2"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        seg = args.cpu_sample_segments
        steps, warm = args.steps, args.warmup
        v, dt, threads, kind = cpu_reference_run(seg, args.points, steps, warm)
        vf, dtf, _, _ = cpu_reference_run(max(1, seg // 2), args.points, 3, 1, full_forward=True)
        sample = f"{seg} segments x {args.points} points per step, {warm} warm-up + {steps} timed ({kind_text(kind)}, encoder, fp32)"
        emit(({
            "impl": "reference", "metric": "segments_per_sec", "value": v, "unit": "segments/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "points_per_sec": v * args.points, "config": config,
            "cpu_baseline": {"value": v, "unit": "segments/s", "cores": threads, "kind": kind, "sample": sample,
                             "full_forward": {"value": vf, "unit": "segments/s", "ms_per_step": dtf * 1e3,
                                              "sample": f"{max(1, seg // 2)} segments x {args.points} points, 1 warm-up + 3 timed, LineRefineNet.forward"}},
            "e2e": {"value": v, "unit": "segments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # ------------------------------------------------------------------ native arm (B200)
    import torch
    import torch.distributed as dist

    import pointnet_refine_b200 as prb
    from pointnet_refine_b200 import _lib, ops      # nothing under oracle/ is imported by the native arm

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    torch.manual_seed(0)                            # random-init weights of the reference architecture (PyTorch default
    model = prb.LineRefineNet()                     # init), BatchNorm affine / running statistics randomised so that the
    with torch.no_grad():                           # folding is not the identity (SURVEY.md section 8d)
        for mod in model.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.normal_(0.0, 0.1)
                mod.running_mean.normal_(0.0, 0.2)
                mod.running_var.uniform_(0.5, 1.5)
    model = model.to(dev).eval()
    model.precision = args.precision
    enc = model.context_encoder
    B, N = args.segments, args.points
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    ctx = torch.randn(B, N, 4, device=dev, generator=gen)

    def step():
        return enc.run_native(ctx, pool=True)["global_feat"]

    extras = {}
    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        launches0 = _lib.launch_counter
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            gf_last = step()
        e1.record()
        barrier()
        launches = _lib.launch_counter - launches0
        clocks = sampler.stop() if rank == 0 else None
        ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
        value = world * B / (ms_per_step * 1e-3)
        if args.dump_outputs and rank == 0:
            dump_global_feat(args.dump_outputs, gf_last)
        del gf_last

        # ---- per-kernel timing for the roofline (same workload, events around every launch)
        prof_steps = min(args.steps, 3)
        ops.profile_enable(True)
        for _ in range(prof_steps):
            step()
        prof = ops.profile_read()
        ops.profile_enable(False)

        # ---- BASELINE configs[3]: training step, 1024 segments x 1024 points per GPU (native train path; FlatDataParallel over
        #      NCCL if N > 1).  Runs ahead of the other extra legs: measured after them, the same step is host-bound on a
        #      multi-rank box (88-190 ms wall for 72 ms of device work), which says nothing about the step itself.
        if not args.no_extras and args.precision == "bf16":
            try:
                with torch.enable_grad():
                    extras["train_step"] = train_step_bench(prb, torch, dist, dev, local_rank, rank, world, barrier, max_over_ranks)
            except torch.cuda.OutOfMemoryError:
                extras["train_step"] = {"error": "out of memory"}
            torch.cuda.empty_cache()

        # ---- HBM roofline of the stand-alone point loader + first layer (north_star evidence item; the bf16 tier's
        #      default path has this stage inside the fused chain kernel): 16 B in + 256 B out per point.  The output
        #      buffer is allocated once and 20 launches are timed back to back; 4M points = 1.1 GB per launch (> L2).
        rows_hbm = min(B * N, 4 * 1024 * 1024)
        folded = enc.folded()
        pts = ctx.reshape(-1, 4)[:rows_hbm]

        def time_embed(tiled):
            out = ops.point_embed(folded, pts, tiled=tiled)
            for _ in range(2):
                ops.point_embed(folded, pts, tiled=tiled, out=out)
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(20):
                ops.point_embed(folded, pts, tiled=tiled, out=out)
            h1.record()
            torch.cuda.synchronize()
            return h0.elapsed_time(h1) / 20
        # bf16 tier: the operand matrix of the default path is tiled (contiguous 16 KB blocks); the row-major figure
        # (128-byte pieces at the 4 KB row pitch, the layout of the tf32 tier) is reported next to it
        embed_ms_rowmajor = time_embed(False)
        embed_ms = time_embed(True) if args.precision == "bf16" else embed_ms_rowmajor
        embed_bytes = rows_hbm * (16 + 2 * 64 * (2 if args.precision == "bf16" else 4))

        # ---- end to end through the module API from pinned host buffers
        host_ctx = torch.empty(B, N, 4, dtype=torch.float32).pin_memory()
        host_ctx.copy_(ctx)
        host_out = torch.empty(B, 2048, dtype=torch.float32).pin_memory()

        from pointnet_refine_b200.stream import HostEncoderPipeline
        pipe = HostEncoderPipeline(enc, segments_per_chunk=512)

        def e2e_step():   # pinned host context -> (chunked H2D overlapped with the encoder) -> pinned host global_feat
            pipe.global_feat(host_ctx, host_out)

        for _ in range(2):
            e2e_step()
        barrier()
        e2e_steps = args.steps
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        e2e_value = world * B / (e2e_ms / e2e_steps * 1e-3)
        del host_ctx, pipe

        if not args.no_extras and args.precision == "bf16":
            # ---- the whole LineRefineNet forward at the configs[1] shape (encoder + context_proj + 6 decoder layers + heads);
            #      the module walks the batch in passes of four encoder waves
            if rank == 0:
                line = torch.randn(B, 32, 3, device=dev, generator=gen)
                model(ctx, line)                     # warm-up at the full shape (allocator, weight preparation)
                torch.cuda.synchronize()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for _ in range(2):
                    out_full = model(ctx, line)
                f1.record()
                torch.cuda.synchronize()
                fm = f0.elapsed_time(f1) * 1e-3 / 2
                extras["full_model"] = {
                    "segments_per_sec": B / fm, "points_per_sec": B * N / fm, "ms_per_forward": fm * 1e3, "segments": B,
                    "points_per_segment": N, "finite": bool(torch.isfinite(out_full).all()),
                    "tflops": (FLOP_PER_POINT_FORWARD * B * N + 0.399e9 * B) / fm / 1e12,
                    "note": "LineRefineNet.forward -> (6,B,32,3) over the whole configs[1] batch (one call, chunked inside the module): "
                            "encoder, context_proj, folded-query cross attention (K/V never materialised) and the query side on the "
                            "sm_100a kernels"}
                del out_full
                if B >= 1024 and B * N >= 1024 * 1024:   # inference_whole_scene.py's setting: 1024 context points per line
                    ctx_ws = ctx.reshape(-1, 4)[:1024 * 1024].view(1024, 1024, 4)
                    for _ in range(2):
                        model(ctx_ws, line[:1024])
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(3):
                        model(ctx_ws, line[:1024])
                    torch.cuda.synchronize()
                    fw = (time.perf_counter() - t0) / 3
                    extras["full_model"]["whole_scene_setting"] = {"segments": 1024, "points_per_segment": 1024, "ms_per_forward": fw * 1e3,
                                                                   "segments_per_sec": 1024 / fw}
                del line

            # ---- BASELINE configs[4]: 256 segments x 65,536 points (same point count as configs[1]; every segment spans 256
            #      tiles and 55 of a wave's CTA pairs, the pooling reduces across tiles, CTAs and waves through atomics)
            if rank == 0 and B * N >= 256 * 65536:
                c5 = ctx.reshape(-1, 4)[:256 * 65536].view(256, 65536, 4)
                enc.run_native(c5, pool=True)
                torch.cuda.synchronize()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for _ in range(3):
                    g5 = enc.run_native(c5, pool=True)["global_feat"]
                f1.record()
                torch.cuda.synchronize()
                t5 = f0.elapsed_time(f1) / 3 * 1e-3
                # property spot checks (no oracle in the native arm): max >= mean >= 0, a segment computed alone gives the same
                # maxima bit for bit, and the means agree to the atomics' summation order
                alone = enc.run_native(c5[7:8].contiguous(), pool=True)["global_feat"]
                extras["config5"] = {
                    "workload": "256 segments x 65,536 points, encoder + max/mean pooling (BASELINE.json configs[4])",
                    "segments_per_sec": 256 / t5, "points_per_sec": 256 * 65536 / t5, "ms_per_pass": t5 * 1e3,
                    "checks": {"finite": bool(torch.isfinite(g5).all()), "max_ge_mean": bool((g5[:, :1024] >= g5[:, 1024:]).all()),
                               "segment_alone_max_bit_equal": bool(torch.equal(alone[0, :1024], g5[7, :1024])),
                               "segment_alone_mean_abs_diff": float((alone[0, 1024:] - g5[7, 1024:]).abs().max())}}
                del c5, g5

            # ---- the other arithmetic tiers on a slice of the same batch (rank 0): tf32 (1e-3 max-abs) and fp32x3 (3 x TF32
            #      split, reproduces the reference's max-pool argmax); roofline against the measured cuBLAS tf32 peak
            if rank == 0:
                peaks_t, _ = load_peaks()
                tf32_pk, tf32_src = tf32_peak(peaks_t)
                tiers = {}
                bt = min(B, 592)
                for tier, passes in (("tf32", 1), ("fp32x3", 3)):
                    model.precision = tier
                    enc.run_native(ctx[:bt], pool=True)
                    torch.cuda.synchronize()
                    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    f0.record()
                    for _ in range(2):
                        gft = enc.run_native(ctx[:bt], pool=True)["global_feat"]
                    f1.record()
                    torch.cuda.synchronize()
                    tt = f0.elapsed_time(f1) / 2 * 1e-3
                    tiers[tier] = {"segments": bt, "segments_per_sec": bt / tt, "points_per_sec": bt * N / tt,
                                   "tensor_tflops": passes * FLOP_PER_POINT_ENCODER * bt * N / tt / 1e12,
                                   "frac_of_tf32_peak": passes * FLOP_PER_POINT_ENCODER * bt * N / tt / 1e12 / tf32_pk,
                                   "finite": bool(torch.isfinite(gft).all())}
                tiers["tf32_peak_tflops"] = tf32_pk
                tiers["tf32_peak_source"] = tf32_src
                tiers["note"] = ("encoder + pooling; tensor_tflops counts the tensor-core passes actually issued (fp32x3: three "
                                 "TF32 passes per k-block)")
                extras["tiers"] = tiers
                model.precision = args.precision
                del gft
                torch.cuda.empty_cache()

            # ---- BASELINE configs[2]: 1M segments x 2048 points over the ranks (strong scaling): every rank pushes a sample of
            #      its shard through the whole forward; inputs are generated on the device chunk by chunk
            total_seg, pts3 = 1_000_000, 2048
            shard_seg = -(-total_seg // world)
            sample_seg = min(shard_seg, 16 * 1184)                      # 16 calls of 1184 segments (two decoder passes each)
            chunk3 = 1184
            ctx3 = torch.randn(chunk3, pts3, 4, device=dev, generator=gen)
            line3 = torch.randn(chunk3, 32, 3, device=dev, generator=gen)
            acc = torch.zeros((), device=dev, dtype=torch.float64)
            model(ctx3, line3)
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            done = 0
            while done < sample_seg:
                n = min(chunk3, sample_seg - done)
                acc.add_(model(ctx3[:n], line3[:n])[-1].double().sum())
                done += n
            f1.record()
            barrier()
            t3 = max_over_ranks(f0.elapsed_time(f1) * 1e-3)
            extras["config3_sample"] = {
                "workload": "inference_whole_scene-style sweep, 1,000,000 segments x 2048 points, LineRefineNet.forward, contiguous segment "
                            "shards over the ranks, no collective (BASELINE.json configs[2])",
                "sample_segments_per_gpu": sample_seg, "shard_segments_per_gpu": shard_seg, "sample_seconds": t3,
                "segments_per_sec": world * sample_seg / t3, "extrapolated_seconds_1M": t3 * shard_seg / sample_seg,
                "finite": bool(torch.isfinite(acc))}
            del ctx3, line3

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_kind = load_peaks()
    f_ms, f_n = prof["fusion"]
    total_ms = sum(v[0] for v in prof.values())
    points_per_launch = B * N * prof_steps / max(f_n, 1)
    achieved = FLOP_PER_POINT_FUSION_KERNEL * points_per_launch / (f_ms / max(f_n, 1) * 1e-3) / 1e12 if f_ms > 0 else 0.0
    peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
    peak_src = f"{peak_kind} bf16_tflops_sustained (cuBLAS 8192^3 back to back under the power cap)"
    if args.precision == "tf32":
        peak, peak_src = tf32_peak(peaks)
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "gemm_pair_kernel<256,EPI_FUSION> (fusion conv + gate + pooling, cta_group::2)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": peak_src,
                # the same kernel time against the burst figure (cuBLAS best of 10, not power-capped): the step's kernels are
                # timed at whatever clock the cap leaves on this box, the sustained figure at a median 1320 MHz
                "frac_of_burst_peak": (achieved / float(peaks["bf16_tflops"])) if args.precision != "tf32" else None,
                "traffic": traffic.get("fusion_dram_bytes_per_launch") if args.precision == "bf16" else None,
                "kernel_ms_per_launch": f_ms / max(f_n, 1), "kernel_share_of_step": f_ms / total_ms if total_ms else None,
                "stage_ms_per_step": {k: v[0] / prof_steps for k, v in prof.items()},
                "whole_encoder_tflops": FLOP_PER_POINT_ENCODER * B * N / (ms_per_step * 1e-3) / 1e12,
                "whole_encoder_frac": FLOP_PER_POINT_ENCODER * B * N / (ms_per_step * 1e-3) / 1e12 / peak}
    # second tensor-bound kernel: the fused conv1..conv5 chain (its tensor-core work = conv2..conv5; contains the
    # widest shared-MLP layer, conv5 512 -> 1024).  bf16 tier only (the tf32 tier runs one kernel per layer).
    c_ms, c_n = prof["conv5"]
    if args.precision == "bf16" and c_n > 0 and c_ms > 0:
        c_ach = FLOP_PER_POINT_CHAIN_KERNEL * B * N * prof_steps / (c_ms * 1e-3) / 1e12
        roofline["chain_kernel"] = {"kernel": "chain_pair_kernel (conv1 FMA + conv2..conv5 on tcgen05, conv5 with A in TMEM)",
                                    "achieved": c_ach, "peak": peak, "unit": "TFLOP/s", "frac": c_ach / peak,
                                    "kernel_ms_per_launch": c_ms / c_n, "kernel_share_of_step": c_ms / total_ms if total_ms else None,
                                    "algorithmic_flop_per_point": FLOP_PER_POINT_CHAIN_KERNEL,
                                    "traffic": traffic.get("chain_dram_bytes_per_launch")}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        seg = args.cpu_sample_segments
        v, dt, threads, kind = cpu_reference_run(seg, N, 5, 1)
        cpu_baseline = {"value": v, "unit": "segments/s", "cores": threads, "kind": kind,
                        "sample": f"{seg} segments x {N} points per step, 1 warm-up + 5 timed ({kind_text(kind)}, encoder, fp32)",
                        "ms_per_step": dt * 1e3}
        v1, dt1, _, _ = cpu_reference_run(2, N, 2, 1, threads=1)       # per-core figure (SURVEY.md section 8d)
        cpu_baseline["single_thread"] = {"value": v1, "cores": 1, "sample": f"2 segments x {N} points per step, 1 warm-up + 2 timed"}
        vf, dtf, _, _ = cpu_reference_run(max(1, seg // 2), N, 2, 1, full_forward=True)
        cpu_baseline["full_forward"] = {"value": vf, "unit": "segments/s", "ms_per_step": dtf * 1e3,
                                        "sample": f"{max(1, seg // 2)} segments x {N} points, 1 warm-up + 2 timed, LineRefineNet.forward"}
        torch.set_num_threads(os.cpu_count() or 1)

    line_out = {
        "metric": "segments_per_sec", "value": value, "unit": "segments/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "points_per_sec": value * N,
        "config": config, "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_value, "unit": "segments/s", "h2d_bytes_per_step": B * N * 16,
                "d2h_bytes_per_step": B * 2048 * 4, "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps},
        "roofline": roofline,
        "roofline_hbm": {"bound": "hbm", "kernel": "point_embed_kernel (point loading + conv1 + gate layer 1, stand-alone)",
                         "achieved": embed_bytes / (embed_ms * 1e-3) / 1e9, "peak": float(peaks["hbm_gbs"]), "unit": "GB/s",
                         "frac": embed_bytes / (embed_ms * 1e-3) / 1e9 / float(peaks["hbm_gbs"]),
                         "traffic": traffic.get("point_embed_dram_bytes_per_launch"),
                         "traffic_points": traffic.get("point_embed_points_per_launch"),
                         "points": rows_hbm, "algorithmic_bytes_per_point": embed_bytes // rows_hbm,
                         "layout": "tiled operand matrix (default bf16 path)" if args.precision == "bf16" else "row-major operand rows",
                         "row_major_achieved": embed_bytes / (embed_ms_rowmajor * 1e-3) / 1e9,
                         "note": "20 launches into one preallocated buffer, events around the loop; the default bf16 path runs this "
                                 "stage inside chain_pair_kernel"},
        "cpu_baseline": cpu_baseline,
    }
    line_out.update(extras)
    emit(line_out)
    if world > 1:
        dist.destroy_process_group()


def train_step_bench(prb, torch, dist, dev, local_rank, rank, world, barrier, max_over_ranks):
    """Forward + L1 deep-supervision loss (train.py:63-69) + backward + Adam at 1024 segments x 1024 points per GPU."""
    from pointnet_refine_b200 import optim as lrn_optim
    Bt, Nt = 1024, 1024
    torch.manual_seed(0)
    m = prb.LineRefineNet().to(dev).train()
    m.context_encoder.native_training = True
    net = m
    if world > 1:     # where train_dist.py:147 wraps the model in DistributedDataParallel: one flat gradient buffer,
        net = prb.FlatDataParallel(m, overlap=os.environ.get("LRN_FDP_OVERLAP", "0") == "1")   # ONE all-reduce of the flat gradient buffer per step
    opt = lrn_optim.FlatAdam(m.parameters(), lr=1e-3, capturable=True)     # step count on the device: the step can be graph-captured
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    ctx = torch.randn(Bt, Nt, 4, device=dev, generator=g)
    line = torch.randn(Bt, 32, 3, device=dev, generator=g)
    tgt = 0.1 * torch.randn(Bt, 32, 3, device=dev, generator=g)

    def one():
        opt.zero_grad()
        loss = lrn_optim.deep_supervision_l1(net(ctx, line), tgt)
        loss.backward()
        opt.step()
        return loss.detach()      # no autograd graph kept alive (its AccumulateGrad nodes would pin this stream at capture time)

    steps = 8

    def timed(fn, warm):
        for _ in range(warm):     # the caching allocator settles within a few steps (a training loop's steady state)
            fn()
        barrier()
        s0 = torch.cuda.memory_stats(dev)
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        clk = sampler.stop() if rank == 0 else None
        s1 = torch.cuda.memory_stats(dev)
        return (max_over_ranks(e0.elapsed_time(e1)) / steps, out, clk,
                int(s1.get("num_device_alloc", 0) - s0.get("num_device_alloc", 0)))

    # (1) the loop body of train.py:56-72 launched from Python, one kernel at a time (~800 launches, ~60 ms of host time)
    eager_ms, loss, eager_clocks, eager_mallocs = timed(one, 4)
    # (2) the same step captured once and replayed (pointnet_refine_b200.GraphedTrainStep): the inputs are copied into the
    #     graph's static buffers inside the timed region; under FlatDataParallel the buffer broadcast and the flat-gradient
    #     all-reduce are nodes of the graph
    ms, clocks, mallocs, mode, graph_note = eager_ms, eager_clocks, eager_mallocs, "eager", None
    if os.environ.get("LRN_BENCH_TRAIN_GRAPH", "1") == "1":
        gstep = None
        try:
            gstep = prb.GraphedTrainStep(net, opt, ctx, line, tgt)
            ms, out, clocks, mallocs = timed(lambda: gstep(ctx, line, tgt), 3)
            loss, mode = out[0].clone(), "cuda_graph_replay"
            del out
        except Exception as e:      # report the eager figure and say why
            graph_note = f"{type(e).__name__}: {e}"[:300]
        finally:
            if gstep is not None:
                gstep.close()       # before destroy_process_group: NCCL waits for graphs that hold its collectives
                del gstep
    allreduce_ms = None
    if world > 1:      # the gradient all-reduce alone: 9,695,954 fp32 = 38.8 MB (what DDP moves per step, train_dist.py:188)
        flat = torch.zeros(9_695_954, device=dev)
        for _ in range(2):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            dist.all_reduce(flat)
        a1.record()
        torch.cuda.synchronize()
        allreduce_ms = max_over_ranks(a0.elapsed_time(a1) / 5)
    diag = None
    if os.environ.get("LRN_BENCH_DIAG") == "1":     # where one more step's time goes (device busy vs collectives vs gaps)
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        per = []
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            one()
            th = time.perf_counter() - t0
            torch.cuda.synchronize()
            per.append((round(th * 1e3, 1), round((time.perf_counter() - t0) * 1e3, 1)))
        print("train_step diag: rank", rank, "(host enqueue ms, step wall ms) x3:", per, file=sys.stderr, flush=True)
        t0 = time.perf_counter()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            one()
            torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ev = prof.key_averages()
        top = sorted(ev, key=lambda e: -e.device_time_total)[:6]
        diag = {"rank": rank, "wall_ms": wall * 1e3, "device_busy_ms": sum(e.device_time_total for e in ev) / 1e3,
                "nccl_ms": sum(e.device_time_total for e in ev if "nccl" in e.key.lower()) / 1e3,
                "top": [(e.key[:60], round(e.device_time_total / 1e3, 2), e.count) for e in top]}
        print("train_step diag:", json.dumps(diag), file=sys.stderr, flush=True)
    peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    return {"workload": "1024 segments x 1024 points per GPU, LineRefineNet train step: forward + L1 deep supervision + backward + Adam "
                        "(BASELINE.json configs[3]); FlatDataParallel (flat gradient buffer, NCCL all-reduce) when n_gpus > 1",
            "ms_per_step": ms, "segments_per_sec": world * Bt / (ms * 1e-3), "n_gpus": world, "allreduce_ms": allreduce_ms,
            "mode": mode, "eager_ms_per_step": eager_ms, "graph_note": graph_note,
            "loss": float(loss.detach()), "finite": bool(torch.isfinite(loss.detach())),
            "bound_ms": TRAIN_BOUND_MS, "frac_of_bound_sustained": TRAIN_BOUND_MS["sustained"] / ms,
            "frac_of_dataflow_floor": TRAIN_BOUND_MS["dataflow"] / ms, "peak_mem_gb": peak_gb,
            "steps": steps, "clocks": clocks, "device_mallocs_in_timed_region": mallocs}


if __name__ == "__main__":
    main()
