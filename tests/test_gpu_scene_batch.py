"""GPU: lines of many scenes in one call (lrn_scenes_segments) and the device-resident training set built on it.
The many-scene call must give, bit for bit, what the per-scene call gives scene by scene and what the oracle gives line by
line under (seeds[l], line_ids[l]); the training set's batches must not depend on which samples share a batch."""
import copy

import numpy as np
import pytest
import torch

from oracle import scene_oracle as so

pytestmark = pytest.mark.gpu

N_MANY, R_MANY = 768, 0.4       # at these settings the scenes below have tubes above N, at or below N, and one empty tube


@pytest.fixture(scope="module")
def dev():
    import pointnet_refine_b200  # noqa: F401  (fails loudly if the library is missing)
    return torch.device("cuda:0")


def _scenes(K, lines_per_scene=None, seed0=100):
    """K synthetic scenes of different sizes and their raw lines; scene 1 (if any) keeps no line, scene 0 gets one extra
    line far from every point (an empty tube)."""
    scenes, lines = [], []
    for k in range(K):
        sc, ln = so.synth_scene(6000 + 5000 * ((k * 7) % 11), lines_per_scene or 2 + k % 3, seed=seed0 + k)
        scenes.append(sc)
        lines.append(ln)
    lines[0] = lines[0] + [lines[0][0] + np.array([0.0, 900.0, 0.0])]
    if K >= 3:
        lines[1] = []
    return scenes, lines


def _interleaved(lines, seed=0):
    """(line_scene, raw lines) with the lines of all scenes shuffled together."""
    items = [(k, raw) for k, ln in enumerate(lines) for raw in ln]
    order = np.random.default_rng(seed).permutation(len(items))
    return np.array([items[i][0] for i in order]), [items[i][1] for i in order]


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("sort", [True, False])
@pytest.mark.parametrize("K", [1, 3, 17])
def test_many_scenes_equal_per_scene_calls_bit_for_bit(dev, K, sort):
    from pointnet_refine_b200 import scene as sc
    scenes, lines = _scenes(K)
    d_scenes = [torch.from_numpy(s).to(dev) for s in scenes]
    prepared = sc.prepare_scenes(d_scenes, sort=sort)
    line_scene, flat = _interleaved(lines, seed=K)
    many = sc.build_segments_many(prepared, flat, line_scene, N_MANY, R_MANY, 2.0, seed=7)
    cnt = many.counts.cpu().numpy()
    assert (cnt > N_MANY).any() and ((cnt > 0) & (cnt <= N_MANY)).any() and (cnt == 0).any()     # all three branches
    for k in range(K):
        rows = np.flatnonzero(line_scene == k)
        if len(rows) == 0:
            continue
        one = sc.build_segments(d_scenes[k], [flat[i] for i in rows], N_MANY, R_MANY, 2.0, seed=7)
        t = torch.from_numpy(rows).to(dev)
        assert torch.equal(_bits(many.context[t]), _bits(one.context)), k
        assert torch.equal(many.indices[t], one.indices) and torch.equal(many.counts[t], one.counts), k
        assert torch.equal(_bits(many.noisy_line[t]), _bits(one.noisy_line)), k
        np.testing.assert_array_equal(many.centers[rows], one.centers)
        np.testing.assert_array_equal(many.line32[rows], one.line32)


def test_many_scenes_equal_oracle_under_per_line_seeds_and_ids(dev):
    from pointnet_refine_b200 import scene as sc
    scenes, lines = _scenes(3, seed0=300)
    prepared = sc.prepare_scenes([torch.from_numpy(s).to(dev) for s in scenes])
    line_scene, flat = _interleaved(lines, seed=5)
    rs = np.random.default_rng(9)
    seeds = rs.integers(0, 2 ** 64 - 1, len(flat), dtype=np.uint64, endpoint=True)
    ids = rs.integers(0, 2 ** 32, len(flat), dtype=np.int64)
    seg = sc.build_segments_many(prepared, flat, line_scene, N_MANY, R_MANY, 2.0, seeds=seeds, line_ids=ids)
    idx, ctx, cnt = seg.indices.cpu().numpy(), seg.context.cpu().numpy(), seg.counts.cpu().numpy()
    noisy = seg.noisy_line.cpu().numpy()
    for l, raw in enumerate(flat):
        o_ctx, o_noisy, o_center, o_idx, o_count = so.build_segment(scenes[line_scene[l]], raw, N_MANY, R_MANY, 2.0,
                                                                    int(seeds[l]), int(ids[l]))
        assert cnt[l] == o_count, (l, cnt[l], o_count)
        np.testing.assert_array_equal(seg.centers[l], o_center)
        np.testing.assert_array_equal(idx[l], o_idx, err_msg=f"line {l}")
        np.testing.assert_array_equal(ctx[l].view(np.uint32), o_ctx.view(np.uint32), err_msg=f"line {l}")
        np.testing.assert_array_equal(noisy[l], o_noisy)


def test_many_scenes_capacity_retry_and_bad_scene_number(dev):
    from pointnet_refine_b200 import scene as sc
    scenes, lines = _scenes(3, seed0=500)
    prepared = sc.prepare_scenes([torch.from_numpy(s).to(dev) for s in scenes])
    line_scene, flat = _interleaved(lines, seed=1)
    a = sc.build_segments_many(prepared, flat, line_scene, 512, 2.0, 2.0, seed=3, capacity=1000)    # far too small: re-run
    b = sc.build_segments_many(prepared, flat, line_scene, 512, 2.0, 2.0, seed=3)
    assert torch.equal(a.indices, b.indices) and torch.equal(_bits(a.context), _bits(b.context)) and torch.equal(a.counts, b.counts)
    with pytest.raises(ValueError):
        sc.build_segments_many(prepared, flat, np.full(len(flat), 3), 512, 2.0, 2.0)                 # checked on the host
    # the library's own check (status[1] bit 2) for a scene number only the device sees
    L = len(flat)
    line32, dense, centers, _, _ = sc._resample_on_device(flat, dev)
    bad = torch.zeros(L, dtype=torch.int32, device=dev)
    bad[L // 2] = 3
    with pytest.raises(ValueError, match="outside"):
        sc.scenes_segments(prepared, bad, dense, line32, centers, torch.zeros(L, dtype=torch.int64, device=dev),
                           torch.arange(L, dtype=torch.int32, device=dev), 512, 2.0, 2.0, 100.0, 1 << 20)


def test_training_batches_equal_per_scene_training_batch(dev):
    from pointnet_refine_b200 import scene as sc
    scenes, lines = _scenes(3, seed0=700)
    d_scenes = [torch.from_numpy(s).to(dev) for s in scenes]
    line_scene, flat = _interleaved(lines, seed=2)
    rs = np.random.default_rng(4)
    gts = [raw + rs.normal(0, 0.2, raw.shape) for raw in flat]
    many = sc.build_training_batches(sc.prepare_scenes(d_scenes), flat, gts, line_scene, 512, 2.0, 2.0, seed=5)
    for k in range(3):
        rows = np.flatnonzero(line_scene == k)
        if len(rows) == 0:
            continue
        one = sc.build_training_batch(d_scenes[k], [flat[i] for i in rows], [gts[i] for i in rows], 512, 2.0, 2.0, seed=5)
        t = torch.from_numpy(rows).to(dev)
        for key in ("context", "noisy_line", "target_offset"):
            assert torch.equal(_bits(many[key][t]), _bits(one[key])), (k, key)


def _training_set(dev, K=4, batch_size=4, seed=0, N=512, r=2.0, **kw):
    from pointnet_refine_b200 import data
    from pointnet_refine_b200 import scene as sc
    scenes, lines = _scenes(K, seed0=900)
    rs = np.random.default_rng(6)
    samples = [(k, raw, raw + rs.normal(0, 0.2, raw.shape)) for k, ln in enumerate(lines) for raw in ln]
    prepared = sc.prepare_scenes([torch.from_numpy(s).to(dev) for s in scenes])
    return data.SceneTrainingSet(prepared, samples, batch_size, N, r, 2.0, seed=seed, **kw), scenes, samples


def test_sample_context_does_not_depend_on_its_batch(dev):
    from pointnet_refine_b200 import data
    ts, scenes, samples = _training_set(dev, seed=11)
    n = len(samples)
    t = lambda *i: torch.tensor(i, dtype=torch.int64, device=dev)   # noqa: E731
    i = 3                                               # a line with points in its tube (sample 2 is the empty one)
    assert samples[i][0] != 0
    alone = ts.batch(t(i), epoch=3)
    first = ts.batch(t(i, 0, n - 1, 5), epoch=3)
    last = ts.batch(t(7, 1, 4, i), epoch=3)
    assert torch.equal(_bits(alone["context"][0]), _bits(first["context"][0]))
    assert torch.equal(_bits(alone["context"][0]), _bits(last["context"][3]))
    assert torch.equal(_bits(alone["target_offset"][0]), _bits(last["target_offset"][3]))
    assert not torch.equal(alone["context"][0], ts.batch(t(i), epoch=4)["context"][0])
    # the draw is the oracle's under (epoch_seed(seed, epoch), sample number)
    for j, row in ((i, alone["context"][0]), (7, last["context"][0])):
        k, raw, _ = samples[j]
        o_ctx = so.build_segment(scenes[k], raw, 512, 2.0, 2.0, data.epoch_seed(11, 3), j)[0]
        np.testing.assert_array_equal(row.cpu().numpy().view(np.uint32), o_ctx.view(np.uint32))


def test_epoch_visits_every_sample_once_and_runs_repeat(dev):
    ts, _, samples = _training_set(dev, batch_size=4, seed=3, drop_last=False)
    again, _, _ = _training_set(dev, batch_size=4, seed=3, drop_last=False)
    ts.set_epoch(2)
    again.set_epoch(2)
    a, b = list(ts), list(again)
    assert len(a) == len(ts) == -(-len(samples) // 4)
    assert sorted(torch.cat([x["sample"] for x in a]).tolist()) == list(range(len(samples)))
    for x, y in zip(a, b):
        assert torch.equal(x["sample"], y["sample"]) and torch.equal(_bits(x["context"]), _bits(y["context"]))
        assert x["context"].shape[1:] == (512, 4) and x["noisy_line"].shape[1:] == (32, 3)
        assert torch.equal(x["target_offset"], ts.target_offset[x["sample"]])
    full, _, _ = _training_set(dev, batch_size=4, seed=3)                   # drop_last: only the partial batch goes
    assert len(list(full)) == len(samples) // 4
    shards = [_training_set(dev, batch_size=2, seed=3, rank=r, world=3, drop_last=False)[0] for r in range(3)]
    seen = [set(torch.cat([x["sample"] for x in s]).tolist()) for s in shards]
    assert set().union(*seen) == set(range(len(samples))) and sum(len(s) for s in seen) == len(samples)


def test_launches_per_batch_do_not_depend_on_the_number_of_scenes(dev):
    from pointnet_refine_b200 import _lib
    ts, _, samples = _training_set(dev, K=18)
    scene_of = np.array([s[0] for s in samples])
    one_scene = torch.from_numpy(np.flatnonzero(scene_of == 0)[:2]).to(dev)
    all_scenes = torch.from_numpy(np.array([np.flatnonzero(scene_of == k)[0] for k in range(18) if (scene_of == k).any()])).to(dev)
    assert len(set(scene_of[all_scenes.cpu().numpy()])) == 17                 # scene 1 has no sample: 17 scenes
    counts = []
    for idx in (one_scene, all_scenes, one_scene, all_scenes):              # first pair: capacity settles
        before = _lib.launch_counter
        ts.batch(idx)
        counts.append(_lib.launch_counter - before)
    assert counts[2] == counts[3], counts


def _no_dropout(m):
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0


def test_training_set_feeds_the_graphed_train_step(dev):
    """GraphedTrainStep built on the first SceneTrainingSet batch replays over the next ones; dropout off, its losses
    follow the eager step fed the same batches (the tolerance of test_gpu_train's graphed-vs-eager check)."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    ts, _, _ = _training_set(dev, batch_size=4, seed=1)
    batches = [(b["context"], b["noisy_line"], b["target_offset"]) for b in ts][:3]
    assert len(batches) >= 2
    torch.manual_seed(0)
    m_g = prb.LineRefineNet().to(dev).train()
    m_g.context_encoder.native_training = True
    _no_dropout(m_g)
    m_e = copy.deepcopy(m_g)
    opt_g, opt_e = FlatAdam(m_g.parameters(), lr=1e-4, capturable=True), FlatAdam(m_e.parameters(), lr=1e-4)
    step = prb.GraphedTrainStep(m_g, opt_g, *batches[0])
    for it in range(6):
        ctx, line, tgt = batches[it % len(batches)]
        loss_g, _ = step(ctx, line, tgt)
        opt_e.zero_grad()
        loss_e = deep_supervision_l1(m_e(ctx, line), tgt)
        loss_e.backward()
        opt_e.step()
        assert np.isfinite(float(loss_g))
        tol = 2e-2 if it < 3 else 6e-2
        assert abs(float(loss_g) - float(loss_e.detach())) <= tol * abs(float(loss_e.detach())), (it, float(loss_g), float(loss_e))
    assert step.replays == 6


def test_refine_scenes_equals_refine_scene_per_scene(dev):
    """bf16 tier, every scene with enough lines that its own forward and the joint one run the decoder in the same regime
    (tensor-core linears, one attention split per segment): bit for bit.  Small scenes: within the tier's tolerance."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200 import scene as sc
    torch.manual_seed(0)
    m = prb.LineRefineNet().to(dev).eval()
    assert m.precision == "bf16"
    big = [so.synth_scene(60_000 + 20_000 * k, 80, seed=40 + k) for k in range(3)]
    d_scenes = [torch.from_numpy(s).to(dev) for s, _ in big] + [torch.from_numpy(big[0][0]).to(dev)]
    lines = [ln for _, ln in big] + [[]]                                     # a scene without lines
    out = sc.refine_scenes(m, d_scenes, lines, 256, 1.0, 2.0, seed=4)
    assert [o.shape for o in out] == [(80, 32, 3)] * 3 + [(0, 32, 3)]
    for k in range(3):
        one = sc.refine_scene(m, d_scenes[k], lines[k], 256, 1.0, 2.0, seed=4)
        np.testing.assert_array_equal(out[k], one, err_msg=f"scene {k}")
    small = [so.synth_scene(30_000, 3, seed=60 + k) for k in range(2)]
    out = sc.refine_scenes(m, [torch.from_numpy(s).to(dev) for s, _ in small], [ln for _, ln in small], 256, 1.0, 2.0, seed=4)
    for k, (s, ln) in enumerate(small):
        one = sc.refine_scene(m, torch.from_numpy(s).to(dev), ln, 256, 1.0, 2.0, seed=4)
        np.testing.assert_allclose(out[k], one, atol=5e-2)
