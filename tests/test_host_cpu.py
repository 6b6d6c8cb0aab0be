"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol the header
declares, the host mirror is state_dict-compatible with the reference interface, argument errors
are raised loudly, and the segment sharding used for N > 1 ranks is exact (gloo, world_size 2)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import pointnet_refine_b200 as prb
from oracle import synth
from pointnet_refine_b200 import _lib, shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol_abi_v3():
    header = open(os.path.join(ROOT, "include", "lrn_b200.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char\*) (lrn_[a-z0-9_]+)\(", header, re.M))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.lrn_abi_version() == _lib.ABI_VERSION == 3
    assert _lib.lib.lrn_status_string(3).decode().startswith("unsupported")
    assert _lib.lib.lrn_encoder_packed_bytes(0) > 2 * 2_803_000 - 700      # bf16 blob holds all matrices
    assert _lib.lib.lrn_encoder_packed_bytes(1) > _lib.lib.lrn_encoder_packed_bytes(0)
    assert _lib.lib.lrn_encoder_packed_bytes(7) == 0
    assert _lib.lib.lrn_encoder_workspace_bytes(0, 10, 0, 1, 0) == 0        # empty input has no workspace


def test_refused_call_enqueues_no_kernel():
    """_lib.launch_counter is the library's own count (lrn_launch_count): a call that validation refuses adds nothing."""
    launches = _lib.launch_counter
    assert _lib.lib.lrn_encoder_forward(None, 0, None, 1, 16, 1, None, None, None, None, 0, None, 0, None) == 6
    assert _lib.launch_counter == launches                                  # a call refused by validation enqueues nothing


def test_packed_layout_mirror_matches_library():
    """The Python copy of the folded blob's layout, which the stage tests read the blob through, totals what the library
    allocates for every tier: a drift of the C++ layout fails here, without a GPU."""
    from tests.test_gpu_encoder_stages import PackedLayout
    for prec, pid in _lib.PRECISIONS.items():
        assert PackedLayout(prec).total == _lib.lib.lrn_encoder_packed_bytes(pid), prec


def test_workspace_layout_mirror_matches_library():
    from tests.test_gpu_encoder_stages import WorkspaceLayout
    flag_sets = (_lib.OUT_POOL, _lib.OUT_ARGMAX, _lib.OUT_FUSED, _lib.OUT_MEMORY, _lib.OUT_POOL | _lib.OUT_ARGMAX,
                 _lib.OUT_FUSED | _lib.OUT_MEMORY, _lib.OUT_POOL | _lib.OUT_ARGMAX | _lib.OUT_FUSED | _lib.OUT_MEMORY,
                 _lib.OUT_MEMORY | _lib.OUT_MEMORY_BF16)
    for B, N in ((1, 1), (1, 127), (3, 1000), (7, 31), (74, 4096), (4096, 4096), (4, 65536)):
        for prec, pid in _lib.PRECISIONS.items():
            for flags in flag_sets:
                for chunk_rows in (0, -1, 1, 127, 128, 129, 128 * 37 * 5, 148 * 128 * 16, 10 ** 8):
                    want = _lib.lib.lrn_encoder_workspace_bytes(B, N, pid, flags, chunk_rows)
                    assert WorkspaceLayout(B, N, prec, flags, chunk_rows).total == want, (B, N, prec, flags, chunk_rows)


def test_state_dict_is_the_reference_tree():
    m = prb.LineRefineNet()
    sd = synth.make_state_dict(0)
    msd = m.state_dict()
    assert list(msd.keys()) == list(sd.keys()) and len(msd) == 205
    for k, v in msd.items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
        assert (v.dtype == torch.int64) == (sd[k].dtype == np.int64), k
    m.load_state_dict(synth.to_torch(sd), strict=True)
    assert sum(p.numel() for p in m.parameters()) == 9_695_954           # SURVEY.md appendix B
    # folded operands / workspaces are caches, never persistent state
    assert not any("fold" in k or "blob" in k for k in msd)


def test_cpu_tensors_fail_loudly():
    m = prb.LineRefineNet().eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU implementation"):
        m(torch.zeros(1, 8, 4), torch.zeros(1, 32, 3))
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU implementation"):
        m.context_encoder(torch.zeros(1, 4, 8))


def test_segment_shard_partitions_exactly():
    for B in (1, 7, 8, 1000, 4096):
        for world in (1, 2, 3, 8):
            got = [i for r in range(world) for i in shard.segment_shard(B, r, world)]
            assert got == list(range(B))
    with pytest.raises(ValueError):
        shard.segment_shard(4, 2, 2)


def _worker(rank, world, port, B, q):
    import torch.distributed as dist
    from oracle import lrn_oracle as orc
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    sd = synth.make_state_dict(0)
    ctx, _ = synth.make_inputs(B, 64, seed=99)
    mine = shard.segment_shard(B, rank, world)
    # the oracle stands in for the device compute here (CPU test of the host-side sharding only)
    gf = orc.encoder_forward(sd, ctx[mine.start:mine.stop])[0] if len(mine) else np.zeros((0, 2048), np.float32)
    full = shard.gather_segments(torch.from_numpy(gf), B)
    if rank == 0:
        q.put(full.numpy())
    dist.destroy_process_group()


def test_sharded_run_equals_unsharded_gloo_world2():
    import torch.multiprocessing as mp
    from oracle import lrn_oracle as orc
    B, world, port = 5, 2, 29541
    ctx_mp = mp.get_context("spawn")
    q = ctx_mp.Queue()
    procs = [ctx_mp.Process(target=_worker, args=(r, world, port, B, q)) for r in range(world)]
    [p.start() for p in procs]
    got = q.get(timeout=120)
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    ctx, _ = synth.make_inputs(B, 64, seed=99)
    want = orc.encoder_forward(synth.make_state_dict(0), ctx)[0]
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)


def test_scene_host_resampling_equals_oracle():
    """The product's polyline resampling (host side of scene.build_segments) and the pinned oracle agree bit for bit."""
    import numpy as np
    from oracle import scene_oracle as so
    from pointnet_refine_b200 import scene as sc
    rs = np.random.default_rng(0)
    for i in range(300):
        nv = int(rs.integers(1, 30))
        pts = np.cumsum(rs.normal(0, 3, (nv, 3)), axis=0) + rs.normal(0, 100, 3)
        if i % 5 == 0 and nv > 3:
            pts[nv // 2] = pts[nv // 2 - 1]                  # a zero-length segment
        for n in (32, 200):
            np.testing.assert_array_equal(sc.resample_polyline(pts, n), so.resample_polyline(pts, n))


def test_compat_shim_resolves_reference_import():
    """`from src.model import LineRefineNet` (reference train.py:7, inference_whole_scene.py:13) resolves to the B200-native
    module when <repo>/compat is ahead on sys.path; the reference's checkpoint round trip
    (torch.save(model.state_dict()) -> load_state_dict(torch.load(..., map_location)), train.py:106 /
    inference_whole_scene.py:203-204) works strictly."""
    import subprocess
    import sys
    code = r"""
import os, sys, tempfile
root = sys.argv[1]
sys.path[:0] = [os.path.join(root, "compat"), root]
import torch
from src.model import LineRefineNet, MultiScalePointNetEncoder, PositionalEncoding, DetrTransformerDecoderLayer
import pointnet_refine_b200 as prb
assert LineRefineNet is prb.LineRefineNet and MultiScalePointNetEncoder is prb.MultiScalePointNetEncoder
model = LineRefineNet()                                   # default-constructed, as every reference script does
assert sum(p.numel() for p in model.parameters()) == 9695954      # the count src/model.py:245 prints
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "best_model.pth")
    torch.save(model.state_dict(), path)
    other = LineRefineNet()
    missing = other.load_state_dict(torch.load(path, map_location="cpu"))      # strict=True is the default
    assert not missing.missing_keys and not missing.unexpected_keys
    for (k, a), (_, b) in zip(model.state_dict().items(), other.state_dict().items()):
        assert torch.equal(a, b), k
enc = MultiScalePointNetEncoder(in_channel=4, out_dim=1024)
assert len(enc.state_dict()) == 46
print("compat ok")
"""
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "compat ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ------------------------------------------------------------------ flat-gradient data parallelism (host logic, gloo)
def _tiny_model():
    import torch.nn as nn

    class Tiny(nn.Module):
        def __init__(self):
            super().__init__()
            self.context_encoder = nn.Sequential(nn.Linear(4, 8), nn.BatchNorm1d(8), nn.ReLU())
            self.head = nn.Linear(8, 2)

        def forward(self, x):
            return self.head(self.context_encoder(x))
    torch.manual_seed(7)
    return Tiny()


def _fdp_worker(rank, world, port, q):
    import torch.distributed as dist
    from pointnet_refine_b200.ddp import FlatDataParallel
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    m = _tiny_model()
    if rank == 1:                                   # replicas must be re-synchronised from rank 0 at wrap time
        with torch.no_grad():
            for p in m.parameters():
                p.add_(1.0)
    net = FlatDataParallel(m, overlap=True)     # two slices: the decoder side as soon as it is complete, the encoder's at the end
    opt = torch.optim.SGD(net.parameters(), lr=0.1)
    x = torch.randn(16, 4, generator=torch.Generator().manual_seed(100 + rank))
    grads = None
    for step in range(2):
        opt.zero_grad()                             # set_to_none: autograd binds fresh .grad tensors, the hooks re-home them
        net(x).square().mean().backward()
        if step == 0:
            grads = [p.grad.clone() for p in m.parameters()]
            assert all(p.grad.data_ptr() == g.data_ptr() for p, g in zip(net.flat.params, net.flat.grad_views))
        opt.step()
    q.put((rank, [g.numpy() for g in grads], [p.detach().numpy().copy() for p in m.parameters()],
           m.context_encoder[1].running_mean.numpy().copy(), net.allreduce_calls))
    dist.destroy_process_group()


def test_flat_data_parallel_two_ranks_gloo():
    """One flat gradient buffer, reduced in two slices (decoder side first, encoder slice at the end of backward):
    gradients equal the mean of the per-rank gradients, replicas stay identical, buffers follow rank 0."""
    import torch.multiprocessing as mp
    world, port = 2, 29547
    ctx_mp = mp.get_context("spawn")
    q = ctx_mp.Queue()
    procs = [ctx_mp.Process(target=_fdp_worker, args=(r, world, port, q)) for r in range(world)]
    [p.start() for p in procs]
    res = dict()
    for _ in range(world):
        r, grads, params, rm, calls = q.get(timeout=180)
        res[r] = (grads, params, rm, calls)
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    # single-process reference: both ranks start from rank 0's weights; gradient = mean over ranks
    want = None
    for rank in range(world):
        m = _tiny_model()
        x = torch.randn(16, 4, generator=torch.Generator().manual_seed(100 + rank))
        m(x).square().mean().backward()
        g = [p.grad.clone() for p in m.parameters()]
        want = g if want is None else [a + b for a, b in zip(want, g)]
    want = [w / world for w in want]
    for rank in range(world):
        for got, w in zip(res[rank][0], want):
            np.testing.assert_allclose(got, w.numpy(), rtol=1e-5, atol=1e-7)
        assert res[rank][3] == 4                    # two slices per step, two steps
    for a, b in zip(res[0][1], res[1][1]):
        assert np.array_equal(a, b)                 # parameters identical after two optimizer steps


def test_thin_linear_split_k_weight_gradient():
    """train_ops.thin_linear (pos_emb.mlp[0] on the polyline points, reg_branches[i][2]): same values and gradients as
    F.linear, with the weight gradient formed as 64 slab products + a sum once there are >= 4096 rows."""
    import torch
    from pointnet_refine_b200.train_ops import thin_linear
    torch.manual_seed(0)
    for rows, fin, fout in ((4096, 3, 256), (4096, 128, 3), (96, 3, 256)):
        x = torch.randn(rows // 32, 32, fin, dtype=torch.float64, requires_grad=True)
        w = torch.randn(fout, fin, dtype=torch.float64, requires_grad=True)
        b = torch.randn(fout, dtype=torch.float64, requires_grad=True)
        r = torch.randn(rows // 32, 32, fout, dtype=torch.float64)
        y = thin_linear(x, w, b)
        ref = torch.nn.functional.linear(x, w, b)
        assert torch.equal(y, ref)
        g = torch.autograd.grad((y * r).sum(), (x, w, b))
        gr = torch.autograd.grad((ref * r).sum(), (x, w, b))
        for a, c in zip(g, gr):
            assert float((a - c).abs().max()) <= 1e-10 * max(1.0, float(c.abs().max()))
