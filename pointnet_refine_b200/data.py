"""Device-resident training set: shuffled training batches drawn from many scenes (DESIGN section 3c).

The reference feeds train.py's loop (train.py:56-72) from `DataLoader(LaneRefineDataset(...))`, which builds every sample
on the host (src/dataset.py:177-253: KD-tree over the 200-point line, query of every scene point, weighted sampling,
normalisation).  `SceneTrainingSet` keeps the scenes and the resampled polylines on the device and builds each batch with
ONE `lrn_scenes_segments` call, whatever the number of scenes its samples come from.  Reading the PCD / JSON files stays
the caller's job: it hands over the scene point clouds and the (scene, noisy polyline, gt polyline) items that
LaneRefineDataset enumerates.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from .scene import (PreparedScenes, _resample_on_device, _seed_bits, _target_offset, default_capacity, prepare_scenes,
                    scenes_segments)

_MASK64 = (1 << 64) - 1


def _splitmix64(x: int) -> int:
    z = (x + 0x9E3779B97F4A7C15) & _MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _MASK64
    return z ^ (z >> 31)


def epoch_seed(seed: int, epoch: int) -> int:
    """The RNG seed of every sample's draw in `epoch` (uint64)."""
    return _splitmix64(_splitmix64(int(seed) & _MASK64) ^ (int(epoch) & _MASK64))


def epoch_order(n: int, seed: int, epoch: int, rank: int = 0, world: int = 1, device="cpu") -> torch.Tensor:
    """This rank's samples of `epoch` in visiting order: a permutation of range(n) from its own torch.Generator seeded from
    (seed, epoch), of which rank r takes entries r, r + world, ... (DistributedSampler's interleaved split, without padding:
    the shards are disjoint and together are the epoch)."""
    if not 0 <= rank < world:
        raise ValueError(f"rank {rank} outside [0, {world})")
    g = torch.Generator(device=device)
    g.manual_seed(epoch_seed(seed, epoch) & ((1 << 63) - 1))
    return torch.randperm(n, generator=g, device=device)[rank::world]


def num_batches(n: int, batch_size: int, world: int = 1, drop_last: bool = True, rank: int = 0) -> int:
    """Batches of a rank per epoch.  drop_last: every rank runs the same number of full batches (what data-parallel
    training needs); otherwise a rank's last batch may be partial and ranks may differ by one batch."""
    if drop_last:
        return (n // world) // batch_size
    shard = len(range(rank, n, world))
    return (shard + batch_size - 1) // batch_size


class SceneTrainingSet:
    """Shuffled training batches of LaneRefineDataset items, built on the device.

    prepared: PreparedScenes (or a list of (S_k, 4) fp32 CUDA scenes); samples: (scene index, noisy polyline, gt polyline)
    per item.  All polylines are resampled once here (dense200, line32, centers, the centred noisy line and target_offset
    stay on the device, indexed by sample).  Per batch: one lrn_scenes_segments call and one host synchronisation (its
    status read); sample i of the set is drawn with seed epoch_seed(seed, epoch) and line id i, so its context depends only
    on (seed, epoch, i), not on which samples share its batch.  Iterating yields {'context' (B,N,4), 'noisy_line' (B,32,3),
    'target_offset' (B,32,3)} fp32 CUDA (build_training_batch's shapes) plus 'sample' (B,) int64, the item numbers.
    set_epoch(e) as DistributedSampler.set_epoch; rank / world: this process's disjoint shard of every epoch."""

    def __init__(self, prepared, samples: Sequence, batch_size: int, num_context_points: int = 2048, crop_radius: float = 4.0,
                 decay_scale: float = 2.0, seed: int = 0, drop_last: bool = True, rank: int = 0, world: int = 1):
        self.prepared = prepared if isinstance(prepared, PreparedScenes) else prepare_scenes(prepared)
        if len(samples) == 0:
            raise ValueError("no samples")
        if batch_size <= 0 or batch_size > 65535:
            raise ValueError(f"batch_size {batch_size} outside [1, 65535]")
        if not 0 <= rank < world:
            raise ValueError(f"rank {rank} outside [0, {world})")
        K = self.prepared.num_scenes
        scene_idx = np.array([int(s[0]) for s in samples], dtype=np.int64)
        if scene_idx.min() < 0 or scene_idx.max() >= K:
            raise ValueError(f"sample scene numbers must lie in [0, {K})")
        dev = self.prepared.points.device
        self.device = dev
        self.n = len(samples)
        self.batch_size, self.drop_last, self.rank, self.world = int(batch_size), bool(drop_last), int(rank), int(world)
        self.num_context_points, self.crop_radius, self.decay_scale = int(num_context_points), float(crop_radius), float(decay_scale)
        self.seed, self.epoch = int(seed), 0
        self.line32, self.dense200, self.centers, self.noisy_line, ext_noisy = _resample_on_device([s[1] for s in samples], dev)
        self.target_offset = _target_offset([s[2] for s in samples], self.line32, self.centers)
        self.line_scene = torch.from_numpy(scene_idx.astype(np.int32)).to(dev)
        self.extent = max(ext_noisy, float(self.prepared.extents.max()))
        self.capacity = default_capacity(int(self.prepared.offsets_host[-1]), self.batch_size, self.num_context_points)

    def set_epoch(self, epoch: int) -> None:
        self.epoch = int(epoch)

    def __len__(self) -> int:
        return num_batches(self.n, self.batch_size, self.world, self.drop_last, self.rank)

    def order(self, epoch: int | None = None) -> torch.Tensor:
        """This rank's sample numbers for the epoch, in visiting order (int64 CUDA)."""
        return epoch_order(self.n, self.seed, self.epoch if epoch is None else epoch, self.rank, self.world, self.device)

    def batch(self, samples: torch.Tensor, epoch: int | None = None) -> dict:
        """The batch of the given sample numbers (int64 CUDA tensor) as drawn in `epoch` (default: the current one)."""
        idx = samples.to(self.device, torch.int64)
        B = int(idx.shape[0])
        seeds = _seed_bits(epoch_seed(self.seed, self.epoch if epoch is None else epoch), B, self.device)
        context, _, _, total = scenes_segments(
            self.prepared, self.line_scene[idx], self.dense200[idx], self.line32[idx], self.centers[idx], seeds,
            idx.to(torch.int32), self.num_context_points, self.crop_radius, self.decay_scale, self.extent, self.capacity)
        if total > self.capacity:                   # the call re-ran at the exact size: keep room for the next batches
            self.capacity = total + total // 4
        return {"context": context, "noisy_line": self.noisy_line[idx], "target_offset": self.target_offset[idx], "sample": idx}

    def __iter__(self):
        order = self.order()
        bs = self.batch_size
        for b in range(len(self)):
            yield self.batch(order[b * bs:(b + 1) * bs])
