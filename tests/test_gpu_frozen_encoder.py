"""Transfer learning on the native path: a frozen context encoder (`context_encoder.eval().requires_grad_(False)` with the
`native_training` opt-in, bf16 tier) runs as its eval forward, whose point-major bf16 `fused` (LRN_OUT_FUSED_BF16) feeds the
native train decoder (`_refine_fast_train`) at M = 32.

The flag's output is checked bit for bit against the fp32 `fused` of LRN_OUT_FUSED rounded to bf16 (both stores round
the same fp32 epilogue value), including the rows past B*N that it must not touch; the frozen step against the stock
decoder on the same frozen encoder (loss and gradient directions, as test_train_native_decoder_close_to_stock does for
the trainable encoder), its routing, its weight caching, its CUDA-graph capture and its launch count."""
import copy
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import synth  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAD_NAMES = ("context_proj.weight", "pos_emb.mlp.2.weight", "decoder_layers.0.cross_attn.in_proj_weight",
              "decoder_layers.5.linear1.weight", "reg_branches.5.0.weight")


@pytest.fixture(scope="module")
def dev():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda:0")


def _model(dev, seed=2):
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev)
    m.load_state_dict(synth.to_torch(synth.make_state_dict(seed)), strict=True)
    return m


def _frozen(m):
    """The transfer-learning recipe: train the model, freeze the encoder, opt in to the native path."""
    m.train()
    m.context_encoder.eval().requires_grad_(False)
    m.context_encoder.native_training = True
    return m


def _no_dropout(m):
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0


def _spy_fast(m):
    calls = []
    fast = m._refine_fast_train
    m._refine_fast_train = lambda *a: calls.append(1) or fast(*a)
    return calls


def _forward_raw(folded, ctx, flags, fused, chunk_rows, prec_id=None):
    """lrn_encoder_forward with a caller-chosen `fused` buffer (or None) and tier (default: the blob's); returns the status."""
    from pointnet_refine_b200 import _lib, ops
    B, N, _ = ctx.shape
    prec_id = folded.prec_id if prec_id is None else prec_id
    nbytes = _lib.lib.lrn_encoder_workspace_bytes(B, N, folded.prec_id, flags, chunk_rows)
    ws = ops._aligned_bytes(max(nbytes, 1024), ctx.device)
    with torch.cuda.device(ctx.device):
        return _lib.lib.lrn_encoder_forward(folded.blob.data_ptr(), prec_id, ctx.data_ptr(), B, N, flags, None,
                                            fused.data_ptr() if fused is not None else None, None, None, chunk_rows,
                                            ws.data_ptr(), ws.numel(), torch.cuda.current_stream(ctx.device).cuda_stream)


# ------------------------------------------------------------------ 1. LRN_OUT_FUSED_BF16 is bf16(LRN_OUT_FUSED)
@pytest.mark.parametrize("B,N", [(3, 700), (7, 300), (1, 129), (4, 1024)])
@pytest.mark.parametrize("chunk_rows", [0, 512])
def test_fused_bf16_is_rounded_fused(dev, B, N, chunk_rows):
    """One wave (default chunk) and many waves (512 rows each), B*N not a multiple of 128 or 256.  The caller's buffer
    is a larger NaN-filled allocation: rows past B*N keep their bits."""
    from pointnet_refine_b200 import _lib, ops
    m = _model(dev).eval()
    enc = m.context_encoder
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=B * 1000 + N)[0]).to(dev)
    fused = ops.encoder_forward(enc.folded(), ctx, pool=False, fused=True, chunk_rows=chunk_rows)["fused"]   # (B,1024,N) fp32
    want = fused.transpose(1, 2).reshape(B * N, 1024).to(torch.bfloat16)
    extra = 300
    buf = torch.full((B * N + extra, 1024), float("nan"), dtype=torch.bfloat16, device=dev)
    poison = buf[B * N:].view(torch.int16).clone()
    assert _forward_raw(enc.folded(proj=False), ctx, _lib.OUT_FUSED_BF16, buf, chunk_rows) == _lib.LRN_OK
    torch.cuda.synchronize()
    assert torch.equal(buf[:B * N].view(torch.int16), want.view(torch.int16))
    assert torch.equal(buf[B * N:].view(torch.int16), poison)
    # the Python entry point, and together with the projection (which then reads the caller's rows): same bits
    out = ops.encoder_forward(enc.folded(proj=False), ctx, pool=False, fused_bf16=True, chunk_rows=chunk_rows)
    assert out["fused_pm"].shape == (B, N, 1024) and out["fused_pm"].dtype == torch.bfloat16
    assert torch.equal(out["fused_pm"].reshape(B * N, 1024).view(torch.int16), want.view(torch.int16))
    both = ops.encoder_forward(enc.folded(), ctx, pool=False, memory=True, memory_bf16=True, fused_bf16=True,
                               chunk_rows=chunk_rows)
    alone = ops.encoder_forward(enc.folded(), ctx, pool=False, memory=True, memory_bf16=True, chunk_rows=chunk_rows)
    assert torch.equal(both["fused_pm"].reshape(B * N, 1024).view(torch.int16), want.view(torch.int16))
    assert torch.equal(both["memory"][..., :256].view(torch.int16), alone["memory"][..., :256].view(torch.int16))


# ------------------------------------------------------------------ 2. refusals
def test_fused_bf16_refusals(dev):
    from pointnet_refine_b200 import _lib, ops
    m = _model(dev).eval()
    enc = m.context_encoder
    B, N = 2, 300
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=3)[0]).to(dev)
    buf = torch.empty(B * N + 8, 1024, dtype=torch.bfloat16, device=dev)
    folded = enc.folded(proj=False)
    F = _lib.OUT_FUSED_BF16
    launches = _lib.launch_counter
    assert _forward_raw(folded, ctx, F | _lib.OUT_FUSED, buf, 0) == 6
    assert _forward_raw(folded, ctx, F, None, 0) == 6
    assert _forward_raw(folded, ctx, F, buf.view(-1)[1:], 0) == 2        # 2-byte offset: not 16-byte aligned
    for prec in (_lib.PREC_TF32, _lib.PREC_FP32X3):      # refused before the blob is read
        assert _forward_raw(folded, ctx, F, buf, 0, prec_id=prec) == 6
    assert _lib.launch_counter == launches
    with pytest.raises(RuntimeError, match="bad argument"):
        ops.encoder_forward(enc.folded(proj=False), ctx, pool=False, fused=True, fused_bf16=True)


# ------------------------------------------------------------------ 3. routing
def test_frozen_encoder_routing(dev):
    """The recipe at M = 32 enters _refine_fast_train; no encoder parameter gets a gradient and the encoder's BatchNorm
    buffers (running statistics, num_batches_tracked) keep their bits over three optimizer steps."""
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    from pointnet_refine_b200.train_ops import native_frozen_encoder, native_train_supported
    m = _frozen(_model(dev))
    enc = m.context_encoder
    assert native_frozen_encoder(enc) and not native_train_supported(enc)
    calls = _spy_fast(m)
    bufs = {k: v.clone() for k, v in enc.state_dict().items()}
    opt = FlatAdam([p for p in m.parameters() if p.requires_grad], lr=1e-3)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    for _ in range(3):
        opt.zero_grad()
        deep_supervision_l1(m(ctx, line), tgt).backward()
        opt.step()
    assert len(calls) == 3
    assert all(p.grad is None for p in enc.parameters())
    assert all(p.grad is not None for n, p in m.named_parameters() if not n.startswith("context_encoder."))
    for k, v in enc.state_dict().items():
        assert torch.equal(v, bufs[k]), k


@pytest.mark.parametrize("case", ["m16", "opt_in_off", "some_bn_frozen", "weights_trainable"])
def test_frozen_encoder_other_cases_keep_their_branch(dev, case):
    from pointnet_refine_b200.train_ops import native_frozen_encoder
    m = _frozen(_model(dev))
    enc = m.context_encoder
    M = 32
    if case == "m16":
        M = 16
    elif case == "opt_in_off":
        enc.native_training = False
    elif case == "some_bn_frozen":                 # encoder in train mode, weights frozen, only bn3 in eval mode
        enc.train()
        enc.bn3.eval()
    else:                                          # BatchNorm frozen, weights trainable: stock ops (out of scope here)
        enc.requires_grad_(True)
    assert native_frozen_encoder(enc) == (case == "m16")
    calls = _spy_fast(m)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(4, 256, M=M, seed=6))
    out = m(ctx, line)
    out.sum().backward()
    assert not calls and out.shape == (6, 4, M, 3) and torch.isfinite(out).all()


# ------------------------------------------------------------------ 4. gradient parity with the stock decoder
@pytest.mark.parametrize("B", [4, 8])
def test_frozen_native_step_close_to_stock(dev, B):
    """Dropout off.  Native arm: the frozen-encoder step (eval encoder's point-major bf16 fused, native train decoder).
    Stock arm: the same frozen encoder's fp32 fused, context_proj, _refine(native_heads=False).  B = 8 (256 query rows)
    also takes the bf16 tensor-core linears on the query side."""
    from pointnet_refine_b200 import ops
    m = _frozen(_model(dev))
    _no_dropout(m)
    calls = _spy_fast(m)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(B, 512, seed=11))
    tgt = 0.1 * torch.randn(B, 32, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    res = {}
    for native in (True, False):
        m.zero_grad()
        if native:
            out = m(ctx, line)
        else:
            _, fused = m.context_encoder(ctx.transpose(2, 1))
            out = m._refine(ctx, line, m.context_proj(fused.transpose(2, 1)), native_heads=False)
        loss = sum(torch.nn.functional.l1_loss(out[l], tgt) for l in range(6)) / 6
        loss.backward()
        res[native] = (float(loss.detach()), {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})
    assert len(calls) == 1
    assert abs(res[True][0] - res[False][0]) <= 2e-2 * abs(res[False][0])
    for n in GRAD_NAMES:
        a, b = res[True][1][n].flatten().double(), res[False][1][n].flatten().double()
        cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
        assert cos >= 0.9, (n, cos)
    assert not any(n.startswith("context_encoder.") for n in res[True][1])
    # both arms' decoders see the same context features: the native arm's fused_pm is bf16 of the stock arm's fused
    fused_pm = ops.encoder_forward(m.context_encoder.folded(proj=False), ctx, pool=False, fused_bf16=True)["fused_pm"]
    assert torch.equal(fused_pm.view(torch.int16), fused.transpose(1, 2).to(torch.bfloat16).view(torch.int16))


# ------------------------------------------------------------------ 5. no re-fold per step
def test_frozen_step_does_not_refold(dev, monkeypatch):
    from pointnet_refine_b200 import ops
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    folds = []

    class Counting(ops.FoldedEncoder):
        def __init__(self, *a, **k):
            folds.append(1)
            super().__init__(*a, **k)
    monkeypatch.setattr(ops, "FoldedEncoder", Counting)
    m = _frozen(_model(dev))
    opt = FlatAdam([p for p in m.parameters() if p.requires_grad], lr=1e-3)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 256, seed=7))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev)
    w0 = m.context_proj.weight.detach().clone()
    blobs = []
    for _ in range(4):
        opt.zero_grad()
        deep_supervision_l1(m(ctx, line), tgt).backward()
        opt.step()
        blobs.append(m._prepared["fold_encoder"][1])
    assert not torch.equal(m.context_proj.weight.detach(), w0)     # context_proj trains ...
    assert len(folds) == 1 and all(b is blobs[0] for b in blobs)    # ... and the encoder was folded once
    assert not blobs[0].has_proj and "fold" not in m._prepared


# ------------------------------------------------------------------ 6. CUDA-graph capture
def test_frozen_graphed_train_step_matches_eager(dev):
    """GraphedTrainStep over the trainable parameters against the eager loop, dropout off: same losses (up to the order of
    fp32 atomics in the decoder's backward), construction leaves the model untouched, the frozen encoder stays frozen,
    the encoder is folded once (not inside the capture) and the step keeps that blob alive."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    torch.manual_seed(0)
    m_g = _frozen(_model(dev))
    _no_dropout(m_g)
    m_e = copy.deepcopy(m_g)
    before = {k: v.clone() for k, v in m_g.state_dict().items()}
    trainable = lambda m: [p for p in m.parameters() if p.requires_grad]
    opt_g, opt_e = FlatAdam(trainable(m_g), lr=1e-4, capturable=True), FlatAdam(trainable(m_e), lr=1e-4)
    batches = []
    for s in range(4):
        ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=20 + s))
        batches.append((ctx, line, 0.1 * torch.randn(8, 32, 3, device=dev)))
    step = prb.GraphedTrainStep(m_g, opt_g, *batches[0])
    for k, v in m_g.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert opt_g.steps_taken == 0
    blob = m_g._prepared["fold_encoder"][1]
    assert step._keep[1]["fold_encoder"][1] is blob
    for it in range(8):
        ctx, line, tgt = batches[it % 4]
        loss_g, _ = step(ctx, line, tgt)
        opt_e.zero_grad()
        loss_e = deep_supervision_l1(m_e(ctx, line), tgt)
        loss_e.backward()
        opt_e.step()
        tol = 2e-2 if it < 3 else 6e-2
        assert abs(float(loss_g) - float(loss_e.detach())) <= tol * abs(float(loss_e.detach())), (it, float(loss_g), float(loss_e))
    assert opt_g.steps_taken == 8 and step.replays == 8
    assert m_g._prepared["fold_encoder"][1] is blob
    sd_g, sd_e = m_g.state_dict(), m_e.state_dict()
    for k, v in sd_g.items():
        if k.startswith("context_encoder."):
            assert torch.equal(v, before[k]), k                     # frozen: weights and BatchNorm buffers untouched
        elif not v.is_floating_point():
            assert torch.equal(v, sd_e[k]), k                       # point_mlp's num_batches_tracked advanced alike
    # the replays moved the parameters as the eager loop did (over all of them: Adam turns the rounding noise of a
    # gradient that is zero in exact arithmetic, e.g. a conv bias ahead of batch-stat BatchNorm, into steps of either sign)
    names = [n for n, p in m_g.named_parameters() if p.requires_grad]
    d_g = torch.cat([(sd_g[n] - before[n]).double().flatten() for n in names])
    d_e = torch.cat([(sd_e[n] - before[n]).double().flatten() for n in names])
    assert float(torch.dot(d_g, d_e) / (d_g.norm() * d_e.norm())) >= 0.9
    m_g.eval(); m_e.eval()
    with torch.no_grad():
        og, oe = m_g(*batches[0][:2]), m_e(*batches[0][:2])
    assert float((og - oe).abs().max()) <= 0.15 * float(oe.abs().max())
    step.close()


def test_frozen_data_parallel_two_ranks_one_gpu():
    """tools/ddp_check.py with the frozen encoder: two ranks on cuda:0 over gloo, DistributedDataParallel and
    FlatDataParallel + FlatAdam over the trainable parameters; gradients identical across ranks and between the wrappers,
    no gradient on the frozen encoder, parameters in sync."""
    env = dict(os.environ, LRN_DDP_BACKEND="gloo", LRN_DDP_ONE_GPU="1", LRN_DDP_FROZEN="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "ddp_check.py"), "8", "512"],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "ddp ok" in r.stdout and '"frozen_encoder": true' in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_frozen_data_parallel_graphed_two_gpus():
    """The same with NCCL on two GPUs, plus a GraphedTrainStep under FlatDataParallel (all-reduce inside the graph)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, LRN_DDP_FROZEN="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tools", "ddp_check.py"), "8", "512"],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "ddp ok" in r.stdout and '"graphed_losses": [' in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ------------------------------------------------------------------ 7. launch count
def test_frozen_step_launch_count(dev):
    """The library's count of one eager frozen step (forward, fused loss, backward, FlatAdam) equals the lrn:: kernels
    the profiler records for it."""
    from torch.profiler import ProfilerActivity, profile
    from pointnet_refine_b200 import _lib
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    m = _frozen(_model(dev))
    opt = FlatAdam([p for p in m.parameters() if p.requires_grad], lr=1e-4, capturable=True)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))

    def step():
        opt.zero_grad()
        deep_supervision_l1(m(ctx, line), tgt).backward()
        opt.step()
    step()                                    # the fold happens here
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        before = _lib.launch_counter
        step()
        torch.cuda.synchronize()
        counted = _lib.launch_counter - before
    names = [e.name for e in prof.events() if "cuda" in str(e.device_type).lower()]
    if not names:
        pytest.skip("the profiler recorded no device activity on this box (CUPTI unavailable)")
    kernels = sum("lrn::" in n for n in names)
    assert counted == kernels > 0, (counted, kernels)
    assert any("chain_pair_kernel" in n for n in names) and not any("bn_finalize_kernel" in n for n in names)   # eval encoder
