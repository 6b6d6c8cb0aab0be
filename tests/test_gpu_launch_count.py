"""The library counts the kernels it enqueues (lrn_launch_count, read as _lib.launch_counter, which bench.py reports as
gpu_launches): for each family of entry points the count one call adds equals the lrn:: / scene:: kernels that a
torch.profiler capture of the same call records on the device."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import synth  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _assert_counted(fn):
    """Runs fn() once under the profiler; the library's count of that call equals its kernels on the device timeline."""
    from torch.profiler import ProfilerActivity, profile
    from pointnet_refine_b200 import _lib
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        before = _lib.launch_counter
        fn()
        torch.cuda.synchronize()
        counted = _lib.launch_counter - before
    names = [e.name for e in prof.events() if "cuda" in str(e.device_type).lower()]
    if not names:
        pytest.skip("the profiler recorded no device activity on this box (CUPTI unavailable)")
    kernels = sum("lrn::" in n or "scene::" in n for n in names)
    assert counted == kernels > 0, (counted, kernels)


def _model(dev, sd_seed=0):
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev)
    m.load_state_dict(synth.to_torch(synth.make_state_dict(sd_seed)), strict=True)
    return m


@pytest.mark.parametrize("proj", [True, False])
def test_fold(dev, proj):
    from pointnet_refine_b200 import ops
    m = _model(dev)
    tensors = {k: v for k, v in m.context_encoder.state_dict().items() if v.is_floating_point()}
    if proj:
        tensors["context_proj.weight"], tensors["context_proj.bias"] = m.context_proj.weight, m.context_proj.bias
    _assert_counted(lambda: ops.FoldedEncoder(tensors, "bf16"))


@pytest.mark.parametrize("prec", ["bf16", "tf32", "fp32x3"])
def test_encoder_forward_several_waves(dev, prec):
    from pointnet_refine_b200 import ops
    m = _model(dev).eval()
    m.precision = prec
    folded = m.context_encoder.folded()
    ctx = torch.from_numpy(synth.make_inputs(3, 700, seed=4)[0]).to(dev)
    run = lambda: ops.encoder_forward(folded, ctx, pool=True, argmax=True, memory=True, chunk_rows=512)   # 5 waves
    run()
    _assert_counted(run)


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
def test_eval_forward(dev, prec):
    m = _model(dev).eval()
    m.precision = prec
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(16, 512, seed=3))
    with torch.no_grad():
        m(ctx, line)                      # weight preparation (folds, uploads) happens on the first call
        _assert_counted(lambda: m(ctx, line))


@pytest.mark.parametrize("point_major", [True, False])
def test_native_train_step(dev, point_major):
    """forward, loss, backward and a capturable FlatAdam step, of the whole model (fused loss; the encoder hands the
    decoder its point-major (B,N,1024) layout) or of the context encoder alone (its channel-major (B,1024,N) layout)."""
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    m = _model(dev, 2).train()
    m.context_encoder.native_training = True
    opt = FlatAdam((m if point_major else m.context_encoder).parameters(), lr=1e-4, capturable=True)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))

    def loss():
        if point_major:
            return deep_supervision_l1(m(ctx, line), tgt)
        global_feat, fused = m.context_encoder(ctx.transpose(2, 1))
        return global_feat.mean() + fused.mean()

    def step():
        opt.zero_grad()
        loss().backward()
        opt.step()
    step()
    _assert_counted(step)


@pytest.mark.parametrize("capacity", [None, 1000])
def test_build_segments(dev, capacity):
    """capacity=1000 is far too small: the crop runs twice (the second time with the exact candidate count)."""
    from oracle import scene_oracle as so
    from pointnet_refine_b200 import scene as sc
    scene, lines = so.synth_scene(60_000, 5, seed=7)
    d_scene = torch.from_numpy(scene).to(dev)
    lines = lines + [lines[0] + np.array([0.0, 900.0, 0.0])]              # a line with an empty tube
    _assert_counted(lambda: sc.build_segments(d_scene, lines, 512, 2.0, 2.0, seed=3, capacity=capacity))
