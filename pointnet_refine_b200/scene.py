"""Whole-scene front end of LineRefineNet on the GPU (SURVEY.md section 8f row 3).

The reference builds the network input for ONE line at a time on the host: KD-tree over a 200-point resampling of the
line, distance query for every scene point, crop, weighted sampling, centroid normalisation
(src/dataset.py:78-130,214-237; inference_whole_scene.py:95-121), then a B = 1 forward per line (:124-142).
`build_segments` does the crop / sampling / normalisation for all lines of a scene in one pass on the device
(`lrn_scene_segments`, csrc/scene_kernels.cuh) and `refine_scene` runs the lines of a scene as one batch.

The polyline resampling runs on the device too (`lrn_scene_resample`, bit-equal to the numpy formulation; the host
`resample_polyline` below is kept for callers and tests).  The draw follows the reproducible RNG contract documented in include/lrn_b200.h (the reference uses the global unseeded
np.random stream): same sampling distribution, fixed by (seed, line number, scene index).
"""
from __future__ import annotations

from typing import NamedTuple, Sequence

import numpy as np
import torch

from ._lib import lib
from .ops import _aligned_bytes, _call


def resample_polyline(points, num_points: int = 32) -> np.ndarray:
    """Arc-length-uniform linear resampling of a polyline (reference src/dataset.py:8-30): float64 (num_points, 3);
    zeros for fewer than two vertices."""
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    if pts.shape[0] < 2:
        return np.zeros((num_points, 3))
    arc = np.concatenate(([0.0], np.cumsum(np.linalg.norm(np.diff(pts, axis=0), axis=1))))
    at = np.linspace(0, arc[-1], num_points)
    return np.column_stack([np.interp(at, arc, pts[:, k]) for k in range(3)])


class PreparedScene(NamedTuple):
    """A scene plus a spatially sorted copy (Morton order of x, y): prepare once, crop many line sets."""
    points: torch.Tensor          # (S, 4) fp32 CUDA, caller's order (what `indices` refer to)
    sorted_points: torch.Tensor   # (S, 4) the same points in Morton order
    perm: torch.Tensor            # (S,) int32: sorted_points[i] = points[perm[i]]
    extent: float                 # largest |coordinate|


def prepare_scene(scene: torch.Tensor, sort: bool = True) -> PreparedScene:
    if not scene.is_cuda or scene.dtype != torch.float32 or scene.dim() != 2 or scene.shape[1] != 4:
        raise TypeError("scene must be a CUDA float32 (S, 4) tensor")
    scene = scene.contiguous()
    if scene.shape[0] == 0:
        raise ValueError("empty scene")
    extent = float(scene[:, :3].abs().max())
    if not sort:
        return PreparedScene(scene, None, None, extent)
    xy = scene[:, :2]
    lo, hi = xy.min(dim=0).values, xy.max(dim=0).values
    q = ((xy - lo) / (hi - lo).clamp_min(1e-6) * 65535.0).to(torch.int64).clamp_(0, 65535)

    def spread(v):   # 16 bits -> every other bit of 32
        v = (v | (v << 8)) & 0x00FF00FF
        v = (v | (v << 4)) & 0x0F0F0F0F
        v = (v | (v << 2)) & 0x33333333
        return (v | (v << 1)) & 0x55555555
    perm = torch.argsort(spread(q[:, 0]) | (spread(q[:, 1]) << 1))
    return PreparedScene(scene, scene[perm].contiguous(), perm.to(torch.int32), extent)


def _resample_on_device(raw_lines: Sequence, dev):
    """Polylines back to back -> one upload -> lrn_scene_resample: (line32 (L,32,3) f64, dense200 (L,200,3) f64,
    centers (L,3) f64, centred line32 (L,32,3) fp32, largest |vertex coordinate|)."""
    L = len(raw_lines)
    arrs = [np.asarray(r, dtype=np.float64).reshape(-1, 3) for r in raw_lines]
    lens = np.fromiter((a.shape[0] for a in arrs), dtype=np.int64, count=L)
    offsets = np.zeros(L + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    verts = np.concatenate(arrs) if offsets[-1] > 0 else np.zeros((1, 3))
    d_verts, d_off = torch.from_numpy(verts).to(dev), torch.from_numpy(offsets).to(dev)
    d_line = torch.empty(L, 32, 3, dtype=torch.float64, device=dev)
    d_dense = torch.empty(L, 200, 3, dtype=torch.float64, device=dev)
    d_cent = torch.empty(L, 3, dtype=torch.float64, device=dev)
    centred = torch.empty(L, 32, 3, dtype=torch.float32, device=dev)
    _call("lrn_scene_resample", dev, d_verts, d_off, L, int(lens.max()), d_line, d_dense, d_cent, centred)
    return d_line, d_dense, d_cent, centred, float(np.abs(verts).max())


class SceneSegments(NamedTuple):
    context: torch.Tensor      # (L, N, 4) fp32 CUDA: sampled points, xyz centred on the line, intensity
    noisy_line: torch.Tensor   # (L, 32, 3) fp32 CUDA: the resampled line, centred
    centers: np.ndarray        # (L, 3) float64 host
    line32: np.ndarray         # (L, 32, 3) float64 host, scene coordinates
    indices: torch.Tensor      # (L, N) int64 CUDA: scene index of every sample, -1 for an empty crop's zero points
    counts: torch.Tensor       # (L,) int32 CUDA: scene points inside each tube


def build_segments(scene, raw_lines: Sequence, num_context_points: int = 1024, crop_radius: float = 0.3,
                   decay_scale: float = 2.0, seed: int = 0, capacity: int | None = None) -> SceneSegments:
    """scene (S, 4) fp32 CUDA [x, y, z, intensity] or a PreparedScene (several line sets over one scene: sort it once);
    raw_lines: polylines (n_i, 3) in scene coordinates.  Defaults are inference_whole_scene.py's (:21-22,
    weighted_sampling's decay_scale); LaneRefineDataset uses 2048 / 4.0 / 2.0."""
    prepared = scene if isinstance(scene, PreparedScene) else prepare_scene(scene)
    scene = prepared.points
    S, L, N = scene.shape[0], len(raw_lines), int(num_context_points)
    if L == 0:
        raise ValueError("no lines")
    dev = scene.device
    d_line, d_dense, d_cent, noisy, extent_lines = _resample_on_device(raw_lines, dev)
    extent = max(extent_lines, prepared.extent)
    context = torch.empty(L, N, 4, dtype=torch.float32, device=dev)
    indices = torch.empty(L, N, dtype=torch.int64, device=dev)
    counts = torch.empty(L, dtype=torch.int32, device=dev)
    status = torch.zeros(2, dtype=torch.int64, device=dev)
    cap = int(capacity) if capacity else max(1 << 20, min(S * L, 8 * L * N))
    for _ in range(2):
        ws = _aligned_bytes(lib.lrn_scene_workspace_bytes(L, cap), dev)
        _call("lrn_scene_segments", dev, scene, S, prepared.sorted_points, prepared.perm,
              d_dense, d_line, d_cent, L, N, float(crop_radius), float(decay_scale), extent, int(seed) & (2 ** 64 - 1), cap,
              context, indices, counts, status, ws, ws.numel())
        total, flags = (int(v) for v in status.tolist())        # synchronises
        if flags & 2:
            raise RuntimeError("lrn_scene_segments: too many candidates tie exactly at a threshold key")
        if not flags & 1:
            break
        cap = total                                                # candidate buffer was too small: exact size now
    else:
        raise RuntimeError("lrn_scene_segments: candidate buffer overflow after resizing")
    return SceneSegments(context, noisy, d_cent.cpu().numpy(), d_line.cpu().numpy(), indices, counts)


def build_training_batch(scene, noisy_lines: Sequence, gt_lines: Sequence, num_context_points: int = 2048,
                         crop_radius: float = 4.0, decay_scale: float = 2.0, seed: int = 0):
    """One scene's training samples as a batch, what LaneRefineDataset.__getitem__ (src/dataset.py:177-253) returns per
    sample: {'context' (L,N,4), 'noisy_line' (L,32,3), 'target_offset' (L,32,3)} fp32 CUDA, with
    target_offset = (gt32 - center) - (noisy32 - center) in float64, rounded once (src/dataset.py:239-243).
    Defaults are LaneRefineDataset's (num_context_points 2048, crop_radius 4.0, decay_scale 2.0)."""
    if len(noisy_lines) != len(gt_lines):
        raise ValueError("one ground-truth polyline per noisy polyline")
    seg = build_segments(scene, noisy_lines, num_context_points, crop_radius, decay_scale, seed)
    dev = seg.context.device
    gt32, _, _, _, _ = _resample_on_device(gt_lines, dev)
    center = torch.from_numpy(seg.centers).to(dev)[:, None, :]
    noisy32 = torch.from_numpy(seg.line32).to(dev)
    target = ((gt32 - center) - (noisy32 - center)).float()
    return {"context": seg.context, "noisy_line": seg.noisy_line, "target_offset": target}


@torch.no_grad()
def refine_scene(model, scene, raw_lines: Sequence, num_context_points: int = 1024, crop_radius: float = 0.3,
                 decay_scale: float = 2.0, seed: int = 0) -> np.ndarray:
    """All lines of a scene through the model in one batch: (L, 32, 3) float64 refined polylines in scene coordinates
    = resampled line + last decoder layer's cumulative offset (inference_whole_scene.py:137-147)."""
    seg = build_segments(scene, raw_lines, num_context_points, crop_radius, decay_scale, seed)
    model.eval()
    offsets = model(seg.context, seg.noisy_line)[-1]
    return seg.line32 + offsets.double().cpu().numpy()
