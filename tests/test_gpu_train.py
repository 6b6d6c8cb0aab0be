"""Train-mode path on the GPU (BASELINE.json configs[3] class): batch-statistic BatchNorm forward and the
hand-written backward through the C ABI (opt-in: `native_training = True`).

Two references:
  * the PARITY reference is the stock-PyTorch fp32 module evaluated on a forward whose tensor-core operands are
    rounded to bf16 at exactly the points where the native path rounds them (`_emulated_encoder`): same ReLU masks,
    same batch statistics, autograd in fp32.  Gradients must agree to 2e-2 relative L2 per parameter.
  * against the un-rounded fp32 module the forward is within 2e-2 of the range; gradients are only required to point
    the same way (cosine), because a bf16 forward flips the ReLU mask of a few per mille of the activations that sit
    at zero (measured 0.4 %) and every flipped element moves its whole gradient.  That is why the native train path
    is opt-in: the default train mode is the reference's fp32 arithmetic."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import synth  # noqa: E402
from tests.golden_util import load_case  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda:0")


def _pair(dev, seed=7):
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev)
    m.load_state_dict(synth.to_torch(synth.make_state_dict(seed)), strict=True)
    enc = m.context_encoder.train()
    ref = copy.deepcopy(enc).train()
    enc.native_training = True             # opt-in: sm_100a train path
    ref.native_training = False            # stock PyTorch ops, fp32
    return enc, ref


def _rb(t):
    """round to bf16, keep fp32 storage; autograd passes the gradient through unchanged"""
    return t.bfloat16().float()


def _saved_activations(node, P):
    """The bf16 activations the native forward kept for its backward (workspace layout of csrc/lrn_abi.cu:train_layout):
    X (P, 2048) = [feat1..feat5 | gate hidden], U (P, 3008) = pre-BatchNorm values of conv1..conv5 and the fusion conv,
    Z (P, 1024) = gate layer 2 pre-activation."""
    ws = node.ws
    Pp = (P + 255) // 256 * 256
    al = lambda v: (v + 1023) // 1024 * 1024
    o_x, o_u = 0, al(Pp * 2048 * 2)
    o_z = o_u + al(Pp * 3008 * 2)
    take = lambda off, cols: ws[off: off + Pp * cols * 2].view(torch.bfloat16).view(Pp, cols)[:P].float()
    return take(o_x, 2048), take(o_u, 3008), take(o_z, 1024)


def _emulated_encoder(ref, ctx, saved=None):
    """Stock fp32 math of MultiScalePointNetEncoder.forward in train mode (src/model.py:39-62) with the operands of every
    tensor-core GEMM and every stored activation rounded to bf16 where csrc/lrn_abi.cu:lrn_encoder_train_forward rounds
    them: U_k (pre-BatchNorm, statistics are taken of the rounded values), X_k, the gate hidden layer, bf16 weights for
    conv2..conv5 / fusion / gate layer 2; conv1 and gate layer 1 consume raw fp32 points.
    `saved` = (X, U, Z) of the native forward: every rounded tensor then takes the native VALUE (which differs from this
    restatement by a bf16 ulp wherever the fp32 accumulation order moved a sum across a rounding boundary) while autograd
    still differentiates the restatement -- identical ReLU masks and batch statistics, fp32 backward."""
    B, N, _ = ctx.shape
    P = B * N
    x = ctx.reshape(P, 4)
    sd = dict(ref.named_parameters())
    w = lambda n: sd[n].squeeze(-1)
    u_off = [0, 64, 192, 448, 960, 1984]
    x_off = [0, 64, 192, 448, 960]

    def pin(t, native):          # value of `native`, gradient of `t`
        return t if native is None else t + (native - t).detach()

    def bn(u, name):
        mu, var = u.mean(0), u.var(0, unbiased=False)
        scale = sd[name + ".weight"] * torch.rsqrt(var + 1e-5)
        return u * scale + (sd[name + ".bias"] - mu * scale)

    X, U, Z = saved if saved is not None else (None, None, None)
    cols = lambda M, o, c: None if M is None else M[:, o:o + c]
    chan = [64, 128, 256, 512, 1024]
    feats = []
    u = pin(_rb(x @ w("conv1.weight").T + sd["conv1.bias"]), cols(U, 0, 64))
    for k in range(1, 6):
        xk = pin(_rb(torch.relu(bn(u, f"bn{k}"))), cols(X, x_off[k - 1], chan[k - 1]))
        feats.append(xk)
        if k < 5:
            u = pin(_rb(xk @ _rb(w(f"conv{k + 1}.weight")).T + sd[f"conv{k + 1}.bias"]), cols(U, u_off[k], chan[k]))
    h = pin(_rb(torch.relu(x[:, 3:4] @ w("intensity_gate.0.weight").T + sd["intensity_gate.0.bias"])), cols(X, 1984, 64))
    uf = pin(_rb(torch.cat(feats, 1) @ _rb(w("fusion.0.weight")).T + sd["fusion.0.bias"]), cols(U, 1984, 1024))
    z = pin(_rb(h @ _rb(w("intensity_gate.2.weight")).T + sd["intensity_gate.2.bias"]), Z)
    fused = torch.relu(bn(uf, "fusion.1")) * (0.5 + 0.5 * torch.sigmoid(z))
    fused = fused.view(B, N, 1024).permute(0, 2, 1)
    return torch.cat([fused.max(dim=2)[0], fused.mean(dim=2)], dim=1), fused


@pytest.mark.parametrize("B,N", [(4, 600), (2, 1024), (8, 2048)])
def test_train_gradients_match_bf16_emulation(dev, B, N):
    """Gradient PARITY of the hand-written backward: fp32 autograd through the restated forward pinned to the native
    forward's own bf16 activations (same masks, same statistics).  What is left is the bf16 rounding of the backward's
    GEMM operands (dY, dU, d feat)."""
    enc, ref = _pair(dev)
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=1241)[0]).to(dev)
    g = torch.Generator(device=dev).manual_seed(3)
    R = torch.randn(B, 1024, N, device=dev, generator=g)
    R2 = torch.randn(B, 2048, device=dev, generator=g)
    gf_n, fz_n = enc(ctx.transpose(2, 1))
    saved = _saved_activations(fz_n.grad_fn, B * N)
    ((fz_n * R).sum() / (B * N) + (gf_n * R2).sum() / B).backward()
    # 1. the restatement on its own reproduces the native forward to a few bf16 ulps of the range
    with torch.no_grad():
        _, fz_free = _emulated_encoder(ref, ctx)
    rng = float(fz_free.abs().max())
    assert float((fz_n.detach() - fz_free).abs().max()) <= 1e-2 * rng
    # 2. pinned to the native activations the fused output agrees to fp32 rounding, and so must the gradients up to
    #    the backward's own bf16 operand rounding
    gf_e, fz_e = _emulated_encoder(ref, ctx, saved)
    assert float((fz_n - fz_e).detach().abs().max()) <= 1e-4 * rng
    ((fz_e * R).sum() / (B * N) + (gf_e * R2).sum() / B).backward()
    worst = {}
    for (name, p), (_, q) in zip(enc.named_parameters(), ref.named_parameters()):
        if name.startswith(("conv", "fusion.0")) and name.endswith("bias"):
            continue                                                        # analytically zero (asserted elsewhere)
        gn, gr = p.grad.flatten().double(), q.grad.flatten().double()
        worst[name] = float((gn - gr).norm() / gr.norm())
    print("train gradient rel-L2 vs fp32 autograd on the native forward state:",
          {k: round(v, 4) for k, v in sorted(worst.items(), key=lambda kv: -kv[1])[:8]})
    bad = {k: v for k, v in worst.items() if v > 2e-2}
    assert not bad, bad


def test_train_statistics_survive_large_means(dev):
    """|mean| >> std in a pre-BatchNorm channel: the statistics are pivot-shifted sums (E[x^2] - mean^2 in fp32 cancels as
    mean^2 / var grows).  conv1's bias is pushed to +-16 while its outputs vary by ~1 (beyond that the bf16 storage of the
    pre-activations, not the statistics, is what limits the batch variance)."""
    enc, ref = _pair(dev)
    with torch.no_grad():
        for e in (enc, ref):
            e.conv1.bias.add_(16.0 * torch.sign(e.conv1.bias))
    ctx = torch.from_numpy(synth.make_inputs(2, 1024, seed=5)[0]).to(dev)
    with torch.no_grad():
        enc(ctx.transpose(2, 1))
        ref(ctx.transpose(2, 1))
    # running_var after one step = 0.9 * old + 0.1 * unbiased batch variance: compare the batch part
    vn, vr = enc.bn1.running_var, ref.bn1.running_var
    assert float(((vn - vr).abs() / vr.abs()).max()) <= 5e-2, float(((vn - vr).abs() / vr.abs()).max())


@pytest.mark.parametrize("B,N", [(4, 600), (2, 1024), (3, 37)])
def test_train_forward_backward_matches_torch(dev, B, N):
    enc, ref = _pair(dev)
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=1241)[0]).to(dev)
    g = torch.Generator(device=dev).manual_seed(3)
    R = torch.randn(B, 1024, N, device=dev, generator=g)
    R2 = torch.randn(B, 2048, device=dev, generator=g)

    def run(e):
        gf, fused = e(ctx.transpose(2, 1))
        ((fused * R).sum() / (B * N) + (gf * R2).sum() / B).backward()
        return gf.detach(), fused.detach()

    gf_r, fz_r = run(ref)
    gf_n, fz_n = run(enc)
    rng = float(fz_r.abs().max())
    assert float((fz_n - fz_r).abs().max()) <= 2e-2 * rng
    assert float((gf_n - gf_r).abs().max()) <= 2e-2 * rng
    # running statistics and the batch counter follow PyTorch's update rule
    for (name, p), (_, q) in zip(enc.named_buffers(), ref.named_buffers()):
        if p.dtype.is_floating_point:
            assert float((p - q).abs().max()) <= 1e-2 * max(float(q.abs().max()), 1e-3), name
        else:
            assert int(p) == int(q) == 1, name
    for (name, p), (_, q) in zip(enc.named_parameters(), ref.named_parameters()):
        assert p.grad is not None and p.grad.shape == q.grad.shape, name
        assert torch.isfinite(p.grad).all(), name
        gn, gr = p.grad.flatten().double(), q.grad.flatten().double()
        if name.startswith(("conv", "fusion.0")) and name.endswith("bias"):
            # a bias in front of a batch-stat BatchNorm has zero gradient (the reference's is fp32 rounding noise of an
            # analytically vanishing sum); the native backward writes the exact zero
            assert float(gn.abs().max()) == 0.0, name
            continue
        cos = float(torch.dot(gn, gr) / (gn.norm() * gr.norm()))
        assert cos >= 0.95, (name, cos)   # direction only: ReLU-mask flips of the bf16 forward (see the module docstring)


def test_train_pooled_loss_uses_native_argmax_scatter(dev):
    """Loss on global_feat only: the backward receives no d_fused at all; the max gradient is scattered to the argmax
    point and the mean gradient spread as 1/N inside the native backward (hand-written backward of src/model.py:58-60)."""
    enc, ref = _pair(dev)
    B, N = 3, 500
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=77)[0]).to(dev)
    R2 = torch.randn(B, 2048, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    res = {}
    for name, e in (("native", enc), ("torch", ref)):
        gf, fused = e(ctx.transpose(2, 1))
        if name == "native":
            assert torch.equal(gf[:, :1024].detach(), fused.detach().max(dim=2)[0])   # pooled in the native forward
            assert float((gf[:, 1024:] - fused.mean(dim=2)).detach().abs().max()) <= 1e-5
        (gf * R2).sum().backward()
        res[name] = {n: p.grad.flatten().double() for n, p in e.named_parameters()}
    for n in ("fusion.0.weight", "fusion.1.weight", "intensity_gate.2.weight", "conv5.weight", "conv3.weight", "bn2.bias"):
        a, b = res["native"][n], res["torch"][n]
        cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
        assert float((a - b).norm() / b.norm()) <= 0.3 and cos >= 0.95, (n, cos)


def test_train_matches_reference_golden(dev):
    """Train-mode forward against the fixture generated from the unmodified reference (oracle/make_golden.py)."""
    g, sd, ctx, _, (sc, sn) = load_case("train_b2_n512")
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev)
    m.load_state_dict(synth.to_torch(sd), strict=True)
    enc = m.context_encoder.train()
    enc.native_training = True
    with torch.no_grad():
        gf, fused = enc(torch.from_numpy(ctx).to(dev).transpose(2, 1))
    rng = max(1.0, float(np.abs(g["global_feat"]).max()))
    assert np.abs(gf.cpu().numpy() - g["global_feat"]).max() <= 2e-2 * rng
    assert np.abs(fused.cpu().numpy()[:, ::sc, ::sn] - g["fused_sub"]).max() <= 2e-2 * rng
    for k, v in enc.state_dict().items():
        ref = g["context_encoder__" + k.replace(".", "__")] if ("running_" in k or "num_batches" in k) else None
        if ref is not None:
            np.testing.assert_allclose(v.cpu().numpy().astype(np.float64), ref, rtol=1e-2, atol=1e-3, err_msg=k)


def test_full_model_train_step_decreases_loss(dev):
    """train.py:56-72 loop body on the native encoder path: loss goes down, every parameter gets a gradient."""
    import pointnet_refine_b200 as prb
    torch.manual_seed(0)
    m = prb.LineRefineNet().to(dev).train()
    m.context_encoder.native_training = True
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev)
    losses = []
    for _ in range(12):
        opt.zero_grad()
        out = m(ctx, line)
        loss = sum(torch.nn.functional.l1_loss(out[l], tgt) for l in range(6)) / 6
        loss.backward()
        assert all(p.grad is not None for p in m.parameters())
        opt.step()
        losses.append(float(loss.detach()))
    assert losses[-1] < losses[0]
    assert int(m.context_encoder.bn1.num_batches_tracked) == 12
    m.eval()
    with torch.no_grad():                       # the eval path re-folds the updated weights and running stats
        assert torch.isfinite(m(ctx, line)).all()


def test_default_train_mode_is_reference_arithmetic(dev):
    """Without the opt-in, model.train() runs the stock fp32 formulation (the reference's numerics); with it, a frozen
    (eval-mode) BatchNorm layer or momentum=None falls back to the stock ops instead of being silently ignored."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.train_ops import native_train_supported
    m = prb.LineRefineNet().to(dev).train()
    assert m.context_encoder.native_training is False
    m.context_encoder.native_training = True
    assert native_train_supported(m.context_encoder)
    m.context_encoder.bn3.eval()
    assert not native_train_supported(m.context_encoder)
    m.context_encoder.bn3.train()
    m.context_encoder.bn2.momentum = None
    assert not native_train_supported(m.context_encoder)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(2, 256, seed=5))
    out = m(ctx, line)                                  # cumulative-average BatchNorm: stock path, still trains
    out.sum().backward()
    assert all(p.grad is not None for p in m.parameters())


def test_ddp_step_two_ranks():
    """train_dist.py-style DDP step (NCCL gradient all-reduce) on the native encoder path; needs 2 GPUs."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", os.path.join(root, "tools", "ddp_check.py"), "8", "512"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ddp ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_data_parallel_step_two_ranks_one_gpu():
    """The same check on a single-GPU box: two ranks share cuda:0 and talk over gloo (NCCL refuses two ranks on one
    device).  Exercises DistributedDataParallel's hooks through the native autograd nodes and FlatDataParallel's flat
    buffers / all-reduce / FlatAdam on the real kernels; gradients identical across ranks and equal between the
    two wrappers, parameters in sync."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, LRN_DDP_BACKEND="gloo", LRN_DDP_ONE_GPU="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29537", os.path.join(root, "tools", "ddp_check.py"), "8", "512"],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "ddp ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_linear_bf16_autograd(dev):
    """The differentiable tensor-core linear used for context_proj / K / V projections in train mode."""
    from pointnet_refine_b200.train_ops import linear_bf16
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(5, 300, 256, device=dev, generator=g, requires_grad=True)
    w = (torch.randn(1536, 256, device=dev, generator=g) / 16).requires_grad_()
    b = torch.randn(1536, device=dev, generator=g, requires_grad=True)
    r = torch.randn(5, 300, 1536, device=dev, generator=g)
    (linear_bf16(x, w, b).float() * r).sum().backward()
    gx, gw, gb = x.grad.clone(), w.grad.clone(), b.grad.clone()
    x.grad = w.grad = b.grad = None
    (torch.nn.functional.linear(x, w, b) * r).sum().backward()
    for a, bb in ((gx, x.grad), (gw, w.grad), (gb, b.grad)):
        assert float((a.float() - bb).norm() / bb.norm()) <= 1e-2


@pytest.mark.parametrize("B", [4, 8])
def test_train_fast_decoder_close_to_stock(dev, B):
    """model.train() with dropout disabled: the tensor-core decoder path gives the same loss and gradients
    (relative L2) as the stock nn.MultiheadAttention formulation on the same native encoder.  B = 8 (256 query rows)
    also takes the bf16 tensor-core linears on the query side."""
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev)
    m.load_state_dict(synth.to_torch(synth.make_state_dict(2)), strict=True)
    m.train()
    m.context_encoder.native_training = True
    for mod in m.modules():                       # switch every dropout off, keep batch-stat BatchNorm
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(B, 512, seed=11))
    tgt = 0.1 * torch.randn(B, 32, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    res = {}
    for fast in (True, False):
        m.fast_decoder = fast
        m.zero_grad()
        out = m(ctx, line)
        loss = sum(torch.nn.functional.l1_loss(out[l], tgt) for l in range(6)) / 6
        loss.backward()
        res[fast] = (float(loss.detach()), {n: p.grad.clone() for n, p in m.named_parameters()})
    assert abs(res[True][0] - res[False][0]) <= 2e-2 * abs(res[False][0])
    for n in ("context_proj.weight", "pos_emb.mlp.2.weight", "decoder_layers.0.cross_attn.in_proj_weight",
              "decoder_layers.5.linear1.weight", "reg_branches.5.0.weight"):
        a, b = res[True][1][n].flatten().double(), res[False][1][n].flatten().double()
        cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
        assert cos >= 0.9, (n, cos)


def test_flat_adam_and_fused_l1_match_torch(dev):
    """FlatAdam (one lrn_adam_step launch over a flat buffer) and deep_supervision_l1 against torch.optim.Adam and the
    reference's loss loop (train.py:40,63-72) over several steps of the same small model."""
    import copy
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    torch.manual_seed(0)
    net_a = torch.nn.Sequential(torch.nn.Linear(96, 64), torch.nn.ReLU(), torch.nn.Linear(64, 6 * 96)).to(dev)
    net_b = copy.deepcopy(net_a)
    opt_a = FlatAdam(net_a.parameters(), lr=1e-3, weight_decay=1e-2)
    opt_b = torch.optim.Adam(net_b.parameters(), lr=1e-3, weight_decay=1e-2)
    x = torch.randn(16, 96, device=dev)
    tgt = torch.randn(16, 32, 3, device=dev)
    for it in range(5):
        losses = []
        for net, opt, fused in ((net_a, opt_a, True), (net_b, opt_b, False)):
            opt.zero_grad()
            pred = net(x).view(16, 6, 32, 3).permute(1, 0, 2, 3)                       # (L, B, M, 3)
            if fused:
                loss = deep_supervision_l1(pred, tgt)
            else:
                loss = sum(torch.nn.functional.l1_loss(pred[l], tgt) for l in range(6)) / 6
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        assert abs(losses[0] - losses[1]) <= 1e-5 * abs(losses[1]), (it, losses)
    for pa, pb in zip(net_a.parameters(), net_b.parameters()):
        assert float((pa - pb).detach().abs().max()) <= 2e-6, float((pa - pb).detach().abs().max())
        assert pa._version > 0


def test_flat_adam_trains_line_refine_net(dev):
    """train.py loop body with FlatAdam + the fused loss on the native train path; eval afterwards re-folds the updated
    weights (the optimizer bumps the parameters' version counters)."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    torch.manual_seed(0)
    m = prb.LineRefineNet().to(dev).train()
    m.context_encoder.native_training = True
    opt = FlatAdam(m.parameters(), lr=1e-3)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev)
    m.eval()
    with torch.no_grad():
        before = m(ctx, line).clone()
    m.train()
    losses = []
    for _ in range(10):
        opt.zero_grad()
        loss = deep_supervision_l1(m(ctx, line), tgt)
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert losses[-1] < losses[0]
    assert len(m.state_dict()) == 205                                        # same checkpoint interface
    m.eval()
    with torch.no_grad():
        after = m(ctx, line)
    assert torch.isfinite(after).all() and float((after - before).abs().max()) > 1e-4


def test_add_layernorm_and_pos_hidden_autograd(dev):
    """Native forward + backward of LayerNorm(x + y) and of the positional hidden layer against stock autograd."""
    from pointnet_refine_b200.train_ops import add_layernorm, pos_hidden_train
    gen = torch.Generator(device=dev).manual_seed(11)
    r = lambda *s: torch.randn(*s, device=dev, generator=gen)
    for rows in (32, 1000, 40000):
        ln = torch.nn.LayerNorm(256).to(dev)
        with torch.no_grad():
            ln.weight.copy_(1 + 0.3 * r(256)); ln.bias.copy_(0.2 * r(256))
        x, y, w = r(rows // 32, 32, 256) * 2 + 0.5, r(rows // 32, 32, 256), r(rows // 32, 32, 256)
        res = []
        for native in (True, False):
            xa, ya = x.clone().requires_grad_(), y.clone().requires_grad_()
            ln.zero_grad()
            out = add_layernorm(xa, ya, ln) if native else ln(xa + ya)
            (out * w).sum().backward()
            res.append((out.detach(), xa.grad, ya.grad, ln.weight.grad.clone(), ln.bias.grad.clone()))
        for a, b in zip(*res):
            assert float((a - b).abs().max()) <= 2e-4 * max(1.0, float(b.abs().max())), rows
    lin = torch.nn.Linear(3, 256).to(dev)
    ctx = r(5, 700, 4)
    wgt = r(5, 700, 256)
    h = pos_hidden_train(ctx, lin.weight, lin.bias)
    assert h.dtype == torch.bfloat16
    (h.float() * wgt).sum().backward()
    gw, gb = lin.weight.grad.clone(), lin.bias.grad.clone()
    lin.zero_grad()
    href = torch.relu(lin(ctx[:, :, :3]))
    (href * wgt.bfloat16().float()).sum().backward()
    assert float((h.float() - href).detach().abs().max()) <= 2 ** -8 * max(1.0, float(href.detach().abs().max()))
    for a, b in ((gw, lin.weight.grad), (gb, lin.bias.grad)):
        assert float((a - b).norm() / b.norm()) <= 1e-2


# ------------------------------------------------------------------ train-mode cross attention (mma.sync kernels)
def _ta_keep_mask(seed, B, N, p, dev):
    """Host mirror of ta_keep_pair (csrc/train_attn.cuh): keep / (1 - p) for element (b*8 + h, query, key); one 32-bit hash
    of the even key's element index decides the even key (low 16 bits) and the odd key (high 16 bits)."""
    M32 = 0xFFFFFFFF
    rows = torch.arange(B * 8 * 32, dtype=torch.int64, device=dev).view(-1, 1)
    keys = torch.arange(N, dtype=torch.int64, device=dev).view(1, -1)
    idx = rows * N + (keys & ~1)
    mul = lambda x, c: (x * c) & M32                       # 32-bit wrap-around product (operands < 2^32: fits int64)
    x = (idx & M32) ^ mul(idx >> 32, 0x85EBCA77) ^ (seed & M32) ^ ((((seed >> 32) & M32) * 0xC2B2AE3D) & M32)
    x = x ^ (x >> 16); x = mul(x, 0x21F0AAAD)
    x = x ^ (x >> 15); x = mul(x, 0x735A2D97)
    x = x ^ (x >> 15)
    bits = torch.where((keys & 1) == 0, x & 0xFFFF, x >> 16)
    keep = bits >= int(p * 65536.0)
    return keep.view(B, 8, 32, N).float() / (1.0 - p)


@pytest.mark.parametrize("B,N,p", [(2, 1024, 0.0), (3, 333, 0.0), (2, 40, 0.1), (2, 1000, 0.1), (2, 333, 0.25)])
def test_train_cross_attention_matches_torch(dev, B, N, p):
    """lrn_train_attention_forward / _backward against the same attention in fp64 on the bf16-rounded operands,
    with the dropout mask regenerated on the host from the kernel's hash; dK / dV land in the shared (B,N,L,H,32) buffers."""
    from pointnet_refine_b200.train_ops import CrossAttnTrainFn, KVGradShare
    g = torch.Generator(device=dev).manual_seed(N)
    L, layer = 6, 4
    q = torch.randn(B, 32, 256, device=dev, generator=g, requires_grad=True)
    kall = torch.randn(B, N, L, 8, 32, device=dev, generator=g).bfloat16().requires_grad_()
    vall = torch.randn(B, N, L, 8, 32, device=dev, generator=g).bfloat16().requires_grad_()
    r = torch.randn(B, 32, 256, device=dev, generator=g)
    share = KVGradShare()
    torch.manual_seed(11)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if p > 0 else 0      # what the Function will draw
    torch.manual_seed(11)
    out = CrossAttnTrainFn.apply(q, kall[:, :, layer].transpose(1, 2), vall[:, :, layer].transpose(1, 2), p, share, layer)
    (out * r).sum().backward()
    # reference in fp64 on the operands the kernel sees (q' and P are rounded to bf16 inside: tolerance covers that)
    qd = q.detach().double().view(B, 32, 8, 32).transpose(1, 2).requires_grad_()
    kd = kall.detach().double()[:, :, layer].transpose(1, 2).requires_grad_()
    vd = vall.detach().double()[:, :, layer].transpose(1, 2).requires_grad_()
    P = torch.softmax(qd @ kd.transpose(2, 3) / 32 ** 0.5, dim=-1)
    if p > 0:
        P = P * _ta_keep_mask(seed, B, N, p, dev).double()
    ref = (P @ vd).transpose(1, 2).reshape(B, 32, 256)
    (ref * r.double()).sum().backward()
    rel = lambda a, b: float((a.detach().double() - b.detach()).norm() / b.detach().norm())
    assert rel(out, ref) <= 1e-2, rel(out, ref)
    assert rel(q.grad, qd.grad.transpose(1, 2).reshape(B, 32, 256)) <= 2e-2
    assert rel(share.dk[:, :, layer], kd.grad.transpose(1, 2)) <= 2e-2
    assert rel(share.dv[:, :, layer], vd.grad.transpose(1, 2)) <= 2e-2
    assert kall.grad is not None and kall.grad.data_ptr() != 0
    assert rel(kall.grad[:, :, layer], kd.grad.transpose(1, 2)) <= 2e-2


def test_train_self_attention_matches_torch(dev):
    """Self attention of the 32 polyline points (N = 32 keys, [q | k] and v with different row pitches) on the same kernels."""
    from pointnet_refine_b200.train_ops import self_attention_train
    g = torch.Generator(device=dev).manual_seed(3)
    B = 5
    qk = torch.randn(B, 32, 512, device=dev, generator=g).bfloat16().requires_grad_()
    v = torch.randn(B, 32, 256, device=dev, generator=g).bfloat16().requires_grad_()
    r = torch.randn(B, 32, 256, device=dev, generator=g)
    out = self_attention_train(qk, v, 0.0)
    (out * r).sum().backward()
    qd = qk.detach().double().requires_grad_()
    vd = v.detach().double().requires_grad_()
    heads = lambda t: t.unflatten(-1, (8, 32)).transpose(1, 2)
    ref = torch.nn.functional.scaled_dot_product_attention(heads(qd[..., :256]), heads(qd[..., 256:]), heads(vd))
    ref = ref.transpose(1, 2).reshape(B, 32, 256)
    (ref * r.double()).sum().backward()
    rel = lambda a, b: float((a.detach().double() - b.detach()).norm() / b.detach().norm())
    assert rel(out, ref) <= 1e-2
    assert rel(qk.grad, qd.grad) <= 2e-2 and rel(v.grad, vd.grad) <= 2e-2


def test_train_attention_seed_state_word(dev):
    """Graph-safe dropout: with train_ops.DropoutSeedState.word installed the kernels use seed = per-call salt + the device
    word (lrn_train_attention_* `seed_state`), forward and backward alike, and a changed word draws a different mask."""
    from pointnet_refine_b200 import train_ops
    from pointnet_refine_b200.train_ops import CrossAttnTrainFn, DropoutSeedState
    B, N, p = 2, 40, 0.25
    g = torch.Generator(device=dev).manual_seed(3)
    q = torch.randn(B, 32, 256, device=dev, generator=g, requires_grad=True)
    k = torch.randn(B, N, 8, 32, device=dev, generator=g).bfloat16().requires_grad_()
    v = torch.randn(B, N, 8, 32, device=dev, generator=g).bfloat16().requires_grad_()
    r = torch.randn(B, 32, 256, device=dev, generator=g)
    word = torch.tensor([123456789012345], dtype=torch.int64, device=dev)
    outs = []
    for w in (123456789012345, 123456789012345, 987654321):
        word.fill_(w)
        DropoutSeedState.word, DropoutSeedState.calls = word, 0
        try:
            for t in (q, k, v):
                t.grad = None
            out = CrossAttnTrainFn.apply(q, k.transpose(1, 2), v.transpose(1, 2), p, None, 0)
            (out * r).sum().backward()
        finally:
            DropoutSeedState.word = None
        outs.append((out.detach().clone(), q.grad.clone(), k.grad.clone()))
    seed = ((1 * 0x9E3779B97F4A7C15) & (2 ** 62 - 1)) + 123456789012345
    qd = q.detach().double().view(B, 32, 8, 32).transpose(1, 2).requires_grad_()
    kd = k.detach().double().transpose(1, 2).requires_grad_()
    vd = v.detach().double().transpose(1, 2)
    P = torch.softmax(qd @ kd.transpose(2, 3) / 32 ** 0.5, dim=-1) * _ta_keep_mask(seed, B, N, p, dev).double()
    ref = (P @ vd).transpose(1, 2).reshape(B, 32, 256)
    (ref * r.double()).sum().backward()
    rel = lambda a, b: float((a.double() - b.detach()).norm() / b.detach().norm())
    assert rel(outs[0][0], ref) <= 1e-2, rel(outs[0][0], ref)
    assert rel(outs[0][1], qd.grad.transpose(1, 2).reshape(B, 32, 256)) <= 2e-2
    assert rel(outs[0][2], kd.grad.transpose(1, 2)) <= 2e-2
    assert torch.equal(outs[0][0], outs[1][0])                       # same word -> same mask
    assert rel(outs[2][0], ref) > 0.1                                # another word -> another mask


def test_flat_adam_capturable_matches_host_step(dev):
    """FlatAdam(capturable=True): the step count and bias corrections live on the device (lrn_adam_step_capturable);
    same trajectory as the host-counted step, and the count round-trips through state_dict."""
    from pointnet_refine_b200.optim import FlatAdam
    torch.manual_seed(0)
    net_a = torch.nn.Linear(96, 64).to(dev)
    net_b = copy.deepcopy(net_a)
    opt_a, opt_b = FlatAdam(net_a.parameters(), lr=1e-3, capturable=True), FlatAdam(net_b.parameters(), lr=1e-3)
    x = torch.randn(16, 96, device=dev)
    for _ in range(7):
        for net, opt in ((net_a, opt_a), (net_b, opt_b)):
            opt.zero_grad()
            net(x).square().mean().backward()
            opt.step()
    for pa, pb in zip(net_a.parameters(), net_b.parameters()):
        assert float((pa - pb).detach().abs().max()) <= 1e-6
    assert opt_a.steps_taken == 7 and opt_a.state_dict()["flat_adam"]["step"] == 7
    opt_c = FlatAdam(copy.deepcopy(net_a).parameters(), lr=1e-3, capturable=True)
    opt_c.load_state_dict(opt_a.state_dict())
    assert opt_c.steps_taken == 7


def _no_dropout(m):
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0


def test_graphed_train_step_matches_eager(dev):
    """GraphedTrainStep (zero_grad -> forward -> loss -> backward -> FlatAdam step as ONE CUDA-graph replay) against the
    same loop run eagerly, dropout off so both are deterministic up to the order of the fp32 atomics: same losses, same
    parameters, BatchNorm counters and Adam step count advance per replay, construction leaves the model untouched."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam, deep_supervision_l1
    torch.manual_seed(0)
    m_g = prb.LineRefineNet().to(dev).train()
    m_g.context_encoder.native_training = True
    _no_dropout(m_g)
    m_e = copy.deepcopy(m_g)
    before = {k: v.clone() for k, v in m_g.state_dict().items()}
    # lr 1e-4: two runs of the SAME loop drift apart step by step (fp32 atomics order feeding bf16 roundings), slowly enough
    # at this rate that eight steps stay comparable
    opt_g, opt_e = FlatAdam(m_g.parameters(), lr=1e-4, capturable=True), FlatAdam(m_e.parameters(), lr=1e-4)
    batches = []
    for s in range(4):
        ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=20 + s))
        batches.append((ctx, line, 0.1 * torch.randn(8, 32, 3, device=dev)))
    step = prb.GraphedTrainStep(m_g, opt_g, *batches[0])
    for k, v in m_g.state_dict().items():                       # warm-up steps were rolled back
        assert torch.equal(v, before[k]), k
    assert opt_g.steps_taken == 0
    for it in range(8):
        ctx, line, tgt = batches[it % 4]
        loss_g, pred_g = step(ctx, line, tgt)
        opt_e.zero_grad()
        pred_e = m_e(ctx, line)
        loss_e = deep_supervision_l1(pred_e, tgt)
        loss_e.backward()
        opt_e.step()
        tol = 2e-2 if it < 3 else 6e-2
        assert abs(float(loss_g) - float(loss_e.detach())) <= tol * abs(float(loss_e.detach())), (it, float(loss_g), float(loss_e.detach()))
    assert opt_g.steps_taken == 8 and int(m_g.context_encoder.bn1.num_batches_tracked) == 8
    assert all(p._version > 0 for p in m_g.parameters())
    m_g.eval(); m_e.eval()
    with torch.no_grad():
        og, oe = m_g(*batches[0][:2]), m_e(*batches[0][:2])
    assert torch.isfinite(og).all()
    assert float((og - oe).abs().max()) <= 0.15 * float(oe.abs().max()), float((og - oe).abs().max())


def test_graphed_train_step_with_dropout_trains(dev):
    """The reference's configuration (dropout 0.1 in the attention weights and the decoder layers): replays draw new
    masks (the seed word advances inside the graph) and the loss goes down."""
    import pointnet_refine_b200 as prb
    from pointnet_refine_b200.optim import FlatAdam
    torch.manual_seed(0)
    m = prb.LineRefineNet().to(dev).train()
    m.context_encoder.native_training = True
    opt = FlatAdam(m.parameters(), lr=1e-3, capturable=True)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 512, seed=5))
    tgt = 0.1 * torch.randn(8, 32, 3, device=dev)
    step = prb.GraphedTrainStep(m, opt, ctx, line, tgt)
    w0 = int(step._seed)
    losses = [float(step(ctx, line, tgt)[0]) for _ in range(12)]
    assert int(step._seed) != w0 and step.replays == 12
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    # a ragged last batch goes through the same step eagerly and shares optimizer state / step count with the replays
    loss_r, pred_r = step(ctx[:5], line[:5], tgt[:5])
    assert pred_r.shape == (6, 5, 32, 3) and bool(torch.isfinite(loss_r)) and step.replays == 12 and opt.steps_taken == 13
    assert np.isfinite(float(step(ctx, line, tgt)[0])) and opt.steps_taken == 14
    step.close()
