"""CPU-only checks of the many-scene front end: its entry points in the header and the library, argument refusal of lrn_scenes_segments, the
per-scene line numbering that reproduces build_segments, and the sampler's epoch order (coverage, determinism, shards)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from pointnet_refine_b200 import _lib, data, scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_scene_entry_points_abi_v4_many_scene_only():
    """ABI version 4: the many-scene entry points are the only scene builders; the per-scene ones are gone everywhere."""
    header = open(os.path.join(ROOT, "include", "lrn_b200.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char\*) (lrn_[a-z0-9_]+)\(", header, re.M))
    many = {"lrn_scenes_segments", "lrn_scenes_workspace_bytes"}
    assert many <= declared and many <= set(_lib.SIGNATURES)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in many:
        assert hasattr(lib, name), name
    for name in ("lrn_scene_segments", "lrn_scene_workspace_bytes"):
        assert name not in header and name not in _lib.SIGNATURES and not hasattr(lib, name), name
    assert lib.lrn_abi_version() == _lib.ABI_VERSION == 4


def test_scenes_workspace_bytes_grow_with_lines_scenes_and_capacity():
    ws = _lib.lib.lrn_scenes_workspace_bytes
    assert ws(0, 3, 100) == 0 and ws(4, 0, 100) == 0 and ws(4, 3, 0) == 0
    base = ws(16, 3, 1 << 20)
    assert ws(16, 3000, 1 << 20) > base and ws(32, 3, 1 << 20) > base and ws(16, 3, 1 << 21) >= base + 12 * (1 << 20)


def _call_scenes(K=2, S=1000, L=4, N=64, capacity=1 << 20, radius=1.0, null=False):
    p = None if null else 1 << 12          # never dereferenced: validation refuses first
    return _lib.lib.lrn_scenes_segments(p, p, K, S, None, None, p, p, p, p, p, p, L, N, radius, 2.0, 10.0, capacity,
                                        p, p, p, p, p, 1 << 30, None)


@pytest.mark.parametrize("kw,status", [
    (dict(null=True), 6),
    (dict(K=0), 1), (dict(K=65536), 1), (dict(L=0), 1), (dict(L=65536), 1), (dict(N=0), 1), (dict(N=4097), 1),
    (dict(S=0), 1), (dict(S=1 << 31), 1), (dict(capacity=0), 1),
    (dict(radius=-1.0), 6),
])
def test_scenes_segments_refuses_bad_arguments_without_launching(kw, status):
    launches = _lib.launch_counter
    assert _call_scenes(**kw) == status
    assert _lib.launch_counter == launches


def test_index_within_scene_numbers_each_scenes_lines_in_order():
    ls = np.array([2, 0, 2, 1, 0, 2, 2, 1])
    np.testing.assert_array_equal(scene.index_within_scene(ls), [0, 0, 1, 0, 1, 2, 3, 1])
    assert scene.index_within_scene([]).shape == (0,)
    rs = np.random.default_rng(0)
    ls = rs.integers(0, 17, 500)
    ids = scene.index_within_scene(ls)
    for k in range(17):
        np.testing.assert_array_equal(ids[ls == k], np.arange((ls == k).sum()))


def test_epoch_seed_depends_on_seed_and_epoch():
    s = {data.epoch_seed(seed, epoch) for seed in range(4) for epoch in range(4)}
    assert len(s) == 16 and all(0 <= v < 2 ** 64 for v in s)
    assert data.epoch_seed(3, 5) == data.epoch_seed(3, 5)


@pytest.mark.parametrize("n,bs", [(100, 7), (96, 8), (5, 8)])
def test_one_epoch_visits_every_sample_once(n, bs):
    order = data.epoch_order(n, seed=1, epoch=0)
    assert sorted(order.tolist()) == list(range(n))
    full = data.num_batches(n, bs, drop_last=True)
    ragged = data.num_batches(n, bs, drop_last=False)
    assert full == n // bs and ragged == -(-n // bs)
    visited = [order[b * bs:(b + 1) * bs].tolist() for b in range(ragged)]
    assert sorted(sum(visited, [])) == list(range(n))
    assert all(len(v) == bs for v in visited[:full])
    kept = sum(visited[:full], [])
    assert len(kept) == n - n % bs and len(set(kept)) == len(kept)                    # drop_last drops only the last partial batch


def test_epoch_order_is_reproducible_and_changes_with_epoch_and_seed():
    a, b = data.epoch_order(500, 7, 3), data.epoch_order(500, 7, 3)
    assert torch.equal(a, b)
    assert not torch.equal(a, data.epoch_order(500, 7, 4))
    assert not torch.equal(a, data.epoch_order(500, 8, 3))


@pytest.mark.parametrize("n,world,bs", [(1000, 4, 16), (1001, 3, 10), (37, 8, 2)])
def test_rank_shards_are_disjoint_and_cover_the_epoch(n, world, bs):
    shards = [data.epoch_order(n, 5, 2, rank=r, world=world) for r in range(world)]
    everything = torch.cat(shards).tolist()
    assert len(everything) == n and sorted(everything) == list(range(n))
    full = data.epoch_order(n, 5, 2)
    for r in range(world):
        assert torch.equal(shards[r], full[r::world])                                # the shards of one shared permutation
    counts = {data.num_batches(n, bs, world, drop_last=True, rank=r) for r in range(world)}
    assert counts == {(n // world) // bs}                                            # same number of steps on every rank
    for r in range(world):
        assert data.num_batches(n, bs, world, drop_last=False, rank=r) * bs >= len(shards[r])
    with pytest.raises(ValueError):
        data.epoch_order(n, 5, 2, rank=world, world=world)
