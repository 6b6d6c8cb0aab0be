"""Whole-scene front end of LineRefineNet on the GPU (SURVEY.md section 8f row 3).

The reference builds the network input for ONE line at a time on the host: KD-tree over a 200-point resampling of the
line, distance query for every scene point, crop, weighted sampling, centroid normalisation
(src/dataset.py:78-130,214-237; inference_whole_scene.py:95-121), then a B = 1 forward per line (:124-142).
`build_segments` does the crop / sampling / normalisation for all lines of a scene in one pass on the device and
`refine_scene` runs the lines of a scene as one batch.  `build_segments_many` / `build_training_batches` / `refine_scenes`
do the same for lines of MANY scenes in one device call over scenes prepared once with `prepare_scenes`.  Every build is
one `lrn_scenes_segments` call (csrc/scene_kernels.cuh); one scene is the case K = 1.  `data.SceneTrainingSet` turns a
set of scenes into shuffled training batches.

The polyline resampling runs on the device too (`lrn_scene_resample`, bit-equal to the numpy formulation; the host
`resample_polyline` below is kept for callers and tests).  The draw follows the reproducible RNG contract documented in include/lrn_b200.h (the reference uses the global unseeded
np.random stream): same sampling distribution, fixed by (seed, line number, scene index).  In the many-scene calls every
line carries its own (seed, line number), and the scene index is the index within that line's scene.
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
    weighted_sampling's decay_scale); LaneRefineDataset uses 2048 / 4.0 / 2.0.  Line l is drawn with (seed, l)."""
    prepared = _one_scene(scene)
    L = len(raw_lines)
    if L == 0:
        raise ValueError("no lines")
    dev = prepared.points.device
    return _segments(prepared, raw_lines, torch.zeros(L, dtype=torch.int32, device=dev), _seed_bits(seed, L, dev),
                     torch.arange(L, dtype=torch.int32, device=dev), num_context_points, crop_radius, decay_scale,
                     float(prepared.extents[0]), capacity)


def build_training_batch(scene, noisy_lines: Sequence, gt_lines: Sequence, num_context_points: int = 2048,
                         crop_radius: float = 4.0, decay_scale: float = 2.0, seed: int = 0):
    """One scene's training samples as a batch, what LaneRefineDataset.__getitem__ (src/dataset.py:177-253) returns per
    sample: {'context' (L,N,4), 'noisy_line' (L,32,3), 'target_offset' (L,32,3)} fp32 CUDA, with
    target_offset = (gt32 - center) - (noisy32 - center) in float64, rounded once (src/dataset.py:239-243).
    Defaults are LaneRefineDataset's (num_context_points 2048, crop_radius 4.0, decay_scale 2.0)."""
    return build_training_batches(_one_scene(scene), noisy_lines, gt_lines, np.zeros(len(noisy_lines), dtype=np.int64),
                                  num_context_points, crop_radius, decay_scale, seed)


@torch.no_grad()
def refine_scene(model, scene, raw_lines: Sequence, num_context_points: int = 1024, crop_radius: float = 0.3,
                 decay_scale: float = 2.0, seed: int = 0) -> np.ndarray:
    """All lines of a scene through the model in one batch: (L, 32, 3) float64 refined polylines in scene coordinates
    = resampled line + last decoder layer's cumulative offset (inference_whole_scene.py:137-147)."""
    seg = build_segments(scene, raw_lines, num_context_points, crop_radius, decay_scale, seed)
    model.eval()
    offsets = model(seg.context, seg.noisy_line)[-1]
    return seg.line32 + offsets.double().cpu().numpy()


# ------------------------------------------------------------------------------------------------ many scenes per call
class PreparedScenes(NamedTuple):
    """K scenes back to back (each with its own Morton-sorted copy): prepare once, build any number of batches from them."""
    points: torch.Tensor          # (S_total, 4) fp32 CUDA, scene k = points[offsets_host[k]:offsets_host[k+1]], caller's order
    offsets: torch.Tensor         # (K+1,) int64 CUDA
    offsets_host: np.ndarray      # (K+1,) int64
    sorted_points: torch.Tensor   # (S_total, 4) every scene in its own Morton order (None: unsorted)
    perm: torch.Tensor            # (S_total,) int32, WITHIN-scene: sorted_points[o_k + i] = points[o_k + perm[o_k + i]]
    extents: np.ndarray           # (K,) largest |coordinate| of every scene

    @property
    def num_scenes(self) -> int:
        return len(self.extents)

    def scene(self, k: int) -> PreparedScene:
        """Scene k as prepare_scene(...) returns it (views into the concatenation)."""
        a, b = int(self.offsets_host[k]), int(self.offsets_host[k + 1])
        if self.sorted_points is None:
            return PreparedScene(self.points[a:b], None, None, float(self.extents[k]))
        return PreparedScene(self.points[a:b], self.sorted_points[a:b], self.perm[a:b], float(self.extents[k]))


def prepare_scenes(scenes: Sequence, sort: bool = True) -> PreparedScenes:
    """(S_k, 4) fp32 CUDA scenes (or PreparedScene) -> PreparedScenes; every scene sorted as prepare_scene sorts it."""
    if len(scenes) == 0:
        raise ValueError("no scenes")
    if len(scenes) > 65535:
        raise ValueError(f"{len(scenes)} scenes: at most 65535 per PreparedScenes")
    preps = [s if isinstance(s, PreparedScene) else prepare_scene(s, sort) for s in scenes]
    dev = preps[0].points.device
    if any(p.points.device != dev for p in preps):
        raise ValueError("all scenes must be on one device")
    sizes = np.array([p.points.shape[0] for p in preps], dtype=np.int64)
    offsets = np.zeros(len(preps) + 1, dtype=np.int64)
    np.cumsum(sizes, out=offsets[1:])
    if offsets[-1] >= 2 ** 31:
        raise ValueError(f"{offsets[-1]} points in all: fewer than 2^31 per PreparedScenes")
    cat = (lambda ts: ts[0]) if len(preps) == 1 else torch.cat      # one scene: its own tensors, not a copy
    points = cat([p.points for p in preps])
    sorted_points = perm = None
    if sort:
        if any(p.sorted_points is None for p in preps):
            raise ValueError("sort=True needs every PreparedScene to carry its sorted copy")
        sorted_points = cat([p.sorted_points for p in preps])
        perm = cat([p.perm for p in preps])
    extents = np.array([p.extent for p in preps], dtype=np.float64)
    return PreparedScenes(points, torch.from_numpy(offsets).to(dev), offsets, sorted_points, perm, extents)


def _host_line_scene(line_scene, L: int, K: int) -> np.ndarray:
    ls = np.asarray(line_scene, dtype=np.int64).reshape(-1)
    if ls.shape[0] != L:
        raise ValueError(f"line_scene has {ls.shape[0]} entries for {L} lines")
    if L and (ls.min() < 0 or ls.max() >= K):
        raise ValueError(f"line_scene must lie in [0, {K})")
    return ls


def index_within_scene(line_scene) -> np.ndarray:
    """Position of every line among the lines of its own scene, in the caller's order: the `line` of the RNG contract
    that build_segments gives each line when it is called once per scene."""
    ls = np.asarray(line_scene, dtype=np.int64).reshape(-1)
    order = np.argsort(ls, kind="stable")
    grouped = ls[order]
    starts = np.flatnonzero(np.r_[True, grouped[1:] != grouped[:-1]]) if len(ls) else np.zeros(0, np.int64)
    run_start = np.repeat(starts, np.diff(np.r_[starts, len(ls)]))
    out = np.empty(len(ls), dtype=np.int64)
    out[order] = np.arange(len(ls)) - run_start
    return out


def _one_scene(scene) -> PreparedScenes:
    """A scene (S, 4) fp32 CUDA, sorted here, or a PreparedScene as a one-scene PreparedScenes over the same tensors."""
    prep = scene if isinstance(scene, PreparedScene) else prepare_scene(scene)
    return prepare_scenes([prep], sort=prep.sorted_points is not None)


def _seed_bits(seeds, L: int, dev) -> torch.Tensor:
    """uint64 seeds as an (L,) int64 CUDA tensor holding the same bits (what the C ABI reads as uint64_t): one seed for
    every line (a device fill) or one per line."""
    if np.ndim(seeds) == 0:
        s = int(seeds) & (2 ** 64 - 1)
        return torch.full((L,), s - 2 ** 64 if s >= 2 ** 63 else s, dtype=torch.int64, device=dev)
    bits = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64)).view(np.int64)
    if bits.shape != (L,):
        raise ValueError("one seed per line")
    return torch.from_numpy(bits).to(dev)


def _target_offset(gt_lines: Sequence, line32: torch.Tensor, centers: torch.Tensor) -> torch.Tensor:
    """LaneRefineDataset's target_offset (src/dataset.py:239-243) of every line: (gt32 - center) - (noisy32 - center) in
    float64, rounded once to fp32; line32 (L,32,3) / centers (L,3) float64 CUDA of the noisy lines."""
    gt32, _, _, _, _ = _resample_on_device(gt_lines, line32.device)
    center = centers[:, None, :]
    return ((gt32 - center) - (line32 - center)).float()


def default_capacity(S: int, L: int, N: int) -> int:
    return max(1 << 20, min(S * L, 8 * L * N))


def scenes_segments(prepared: PreparedScenes, line_scene: torch.Tensor, dense200: torch.Tensor, line32: torch.Tensor,
                    centers: torch.Tensor, seeds: torch.Tensor, line_ids: torch.Tensor, num_context_points: int,
                    crop_radius: float, decay_scale: float, extent: float, capacity: int):
    """lrn_scenes_segments on device inputs (line_scene (L,) int32, seeds (L,) int64 bits of uint64, line_ids (L,) int32,
    resampled lines as lrn_scene_resample writes them) -> (context, indices, counts, total candidates).  One status read;
    a second call only when `capacity` was too small (then with the exact size)."""
    dev = prepared.points.device
    K, S = prepared.num_scenes, int(prepared.offsets_host[-1])
    L, N = int(line_scene.shape[0]), int(num_context_points)
    if L == 0:
        raise ValueError("no lines")
    context = torch.empty(L, N, 4, dtype=torch.float32, device=dev)
    indices = torch.empty(L, N, dtype=torch.int64, device=dev)
    counts = torch.empty(L, dtype=torch.int32, device=dev)
    status = torch.zeros(2, dtype=torch.int64, device=dev)
    cap = int(capacity)
    for _ in range(2):
        ws = _aligned_bytes(lib.lrn_scenes_workspace_bytes(L, K, cap), dev)
        _call("lrn_scenes_segments", dev, prepared.points, prepared.offsets, K, S, prepared.sorted_points, prepared.perm,
              line_scene, dense200, line32, centers, seeds, line_ids, L, N, float(crop_radius), float(decay_scale),
              float(extent), cap, context, indices, counts, status, ws, ws.numel())
        total, flags = (int(v) for v in status.tolist())        # synchronises
        if flags & 4:
            raise ValueError(f"lrn_scenes_segments: a line's scene number is outside [0, {K})")
        if flags & 2:
            raise RuntimeError("lrn_scenes_segments: too many candidates tie exactly at a threshold key")
        if not flags & 1:
            return context, indices, counts, total
        cap = total                                                # candidate buffer was too small: exact size now
    raise RuntimeError("lrn_scenes_segments: candidate buffer overflow after resizing")


def build_segments_many(prepared, raw_lines: Sequence, line_scene, num_context_points: int = 1024, crop_radius: float = 0.3,
                        decay_scale: float = 2.0, seed: int = 0, seeds=None, line_ids=None,
                        capacity: int | None = None) -> SceneSegments:
    """build_segments for lines of many scenes in ONE device call.  prepared: PreparedScenes (or a list of scenes);
    raw_lines: polylines (n_i, 3) in the coordinates of their scene; line_scene: scene number of every line (lines of
    different scenes may be interleaved).  Outputs are in the caller's line order and `indices` are within each line's scene.
    The draw of line l is fixed by (seeds[l], line_ids[l]); the defaults (seed for every line, line_ids = position of the
    line among its scene's lines) give exactly what build_segments(scene_k, lines of k, ..., seed) gives scene by scene."""
    prepared = prepared if isinstance(prepared, PreparedScenes) else prepare_scenes(prepared)
    L, K = len(raw_lines), prepared.num_scenes
    if L == 0:
        raise ValueError("no lines")
    ls = _host_line_scene(line_scene, L, K)
    dev = prepared.points.device
    line_ids = index_within_scene(ls) if line_ids is None else np.asarray(line_ids, dtype=np.int64)
    if line_ids.shape != (L,):
        raise ValueError("one line id per line")
    if line_ids.min() < 0 or line_ids.max() >= 2 ** 32:
        raise ValueError("line ids are uint32")
    return _segments(prepared, raw_lines, torch.from_numpy(ls.astype(np.int32)).to(dev),
                     _seed_bits(seed if seeds is None else seeds, L, dev),
                     torch.from_numpy(line_ids.astype(np.uint32).view(np.int32)).to(dev), num_context_points, crop_radius,
                     decay_scale, float(prepared.extents[np.unique(ls)].max()), capacity)


def _segments(prepared: PreparedScenes, raw_lines: Sequence, line_scene, seeds, line_ids, num_context_points, crop_radius,
              decay_scale, extent: float, capacity) -> SceneSegments:
    """The lines resampled on the device, then scenes_segments over them; extent: of the scenes the lines lie in."""
    d_line, d_dense, d_cent, noisy, extent_lines = _resample_on_device(raw_lines, prepared.points.device)
    N = int(num_context_points)
    cap = int(capacity) if capacity else default_capacity(int(prepared.offsets_host[-1]), len(raw_lines), N)
    context, indices, counts, _ = scenes_segments(prepared, line_scene, d_dense, d_line, d_cent, seeds, line_ids, N, crop_radius,
                                                  decay_scale, max(extent, extent_lines), cap)
    return SceneSegments(context, noisy, d_cent.cpu().numpy(), d_line.cpu().numpy(), indices, counts)


def build_training_batches(prepared, noisy_lines: Sequence, gt_lines: Sequence, line_scene, num_context_points: int = 2048,
                           crop_radius: float = 4.0, decay_scale: float = 2.0, seed: int = 0, seeds=None, line_ids=None):
    """build_training_batch for samples of many scenes in one device call, in the caller's order: {'context' (L,N,4),
    'noisy_line' (L,32,3), 'target_offset' (L,32,3)} fp32 CUDA.  Seeds and line ids as in build_segments_many (the defaults
    give build_training_batch per scene).  Defaults are LaneRefineDataset's (2048 / 4.0 / 2.0)."""
    if len(noisy_lines) != len(gt_lines):
        raise ValueError("one ground-truth polyline per noisy polyline")
    seg = build_segments_many(prepared, noisy_lines, line_scene, num_context_points, crop_radius, decay_scale, seed, seeds,
                              line_ids)
    dev = seg.context.device
    target = _target_offset(gt_lines, torch.from_numpy(seg.line32).to(dev), torch.from_numpy(seg.centers).to(dev))
    return {"context": seg.context, "noisy_line": seg.noisy_line, "target_offset": target}


@torch.no_grad()
def refine_scenes(model, prepared, lines_per_scene: Sequence[Sequence], num_context_points: int = 1024,
                  crop_radius: float = 0.3, decay_scale: float = 2.0, seed: int = 0) -> list:
    """refine_scene for many scenes (inference_whole_scene.py's loop over scene files): one build_segments_many call and
    one model forward over all lines (the model splits it into its own chunks).  lines_per_scene[k] are scene k's
    polylines; returns one (L_k, 32, 3) float64 array per scene.  The segments are those refine_scene builds per scene; the
    offsets are bit-identical to refine_scene's where both forwards run the decoder in the same regime (DESIGN section 3c)."""
    prepared = prepared if isinstance(prepared, PreparedScenes) else prepare_scenes(prepared)
    if len(lines_per_scene) != prepared.num_scenes:
        raise ValueError(f"{len(lines_per_scene)} line lists for {prepared.num_scenes} scenes")
    sizes = [len(lines) for lines in lines_per_scene]
    flat = [line for lines in lines_per_scene for line in lines]
    if not flat:
        return [np.zeros((0, 32, 3)) for _ in sizes]
    line_scene = np.repeat(np.arange(len(sizes)), sizes)
    seg = build_segments_many(prepared, flat, line_scene, num_context_points, crop_radius, decay_scale, seed)
    model.eval()
    refined = seg.line32 + model(seg.context, seg.noisy_line)[-1].double().cpu().numpy()
    return np.split(refined, np.cumsum(sizes)[:-1])
