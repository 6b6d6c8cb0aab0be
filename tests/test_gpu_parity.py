"""GPU parity tests (run with -m gpu on a B200).  Everything goes through the C ABI
(pointnet_refine_b200.ops -> liblrn_b200.so); the numpy oracle and the committed golden fixtures
(generated from the unmodified reference, oracle/make_golden.py) are the checkers.

Tolerances (north_star), for the global feature AND the refined offsets: TF32 tier max-abs 1e-3; bf16 tier 1e-2
relative to the output range.  argmax: bit-exact wherever the reference's top-2 gap exceeds twice the tier's value
tolerance; over ALL untied (segment, channel) pairs the agreement rate is measured, reported
(gpurun_out/parity_report.jsonl) and held above a floor per tier (reduced-precision operands cannot reproduce an
argmax whose top-2 gap is below their rounding error, SURVEY.md section 7.3).

Accepted argmax deviation, spelled out: north_star asks for bit-exact indices "where the reference has no ties".
bf16 / tf32 tiers: exact equality is asserted only on the gap-filtered subset; on the remaining untied pairs (gap > 0
but within 2x tolerance) indices may differ from the reference, bounded by the agreement floors below.  fp32x3 tier
(LRN_PREC_FP32X3, `model.precision = "fp32x3"`): exact equality on ALL untied pairs, i.e. what north_star states."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import lrn_oracle as orc  # noqa: E402
from oracle import synth  # noqa: E402
from tests.golden_util import EVAL_CASES, load_case, report  # noqa: E402

TIERS = {"bf16": 1e-2, "tf32": 1e-3, "fp32x3": 1e-4}      # fp32x3: 3 x TF32 split (fp32-class products; see DESIGN.md section 4)
# floor of the argmax agreement with the fp32 reference over ALL untied (segment, channel) pairs.  Measured on the
# B200 (gpurun_out/parity_report.jsonl -> profiles/r02_parity_report.jsonl): bf16 98.9-99.3 % on the N(0,1) fixtures and
# 95.3 % on the realistic one (x up to +-25 m, value range 10), tf32 99.86-100 %; SURVEY.md section 7.3 predicted
# 98.1-98.9 % / 99.7-99.9 % from a CPU emulation of the operand rounding.  The opt-in fp32x3 tier (3 x TF32 split, gate in
# full fp32) reproduces the reference's argmax on EVERY untied pair of every fixture (13-14k pairs), which is asserted.
ARGMAX_FLOOR = {"bf16": 0.94, "tf32": 0.995, "fp32x3": 1.0}   # fp32x3: every untied pair of every fixture (measured 100 %)


def _offset_tol(prec, ref_out):
    """north_star: refined offsets within 1e-2 of their range (bf16 tier) / 1e-3 max-abs (tf32 tier); fp32x3: 1e-4."""
    return {"bf16": 1e-2 * max(1.0, float(np.abs(ref_out).max())), "tf32": 1e-3, "fp32x3": 1e-4}[prec]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cudnn.allow_tf32 = False       # keep the stock-PyTorch decoder in true fp32 for parity
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda:0")


def _model(sd, dev, prec):
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev).eval()
    m.load_state_dict(synth.to_torch(sd), strict=True)
    m.precision = prec
    return m


# ------------------------------------------------------------------ building block
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (300, 128, 128), (1000, 256, 512), (5000, 1024, 512), (129, 512, 256)])
def test_gemm_bf16_matches_fp64(dev, M, N, K):
    from pointnet_refine_b200 import ops
    g = torch.Generator(device=dev).manual_seed(M + N + K)
    a = torch.randn(M, K, device=dev, generator=g).bfloat16()
    w = (torch.randn(N, K, device=dev, generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device=dev, generator=g)
    out = ops.gemm_bias_act(a, w, b, relu=True, out_dtype=torch.float32)
    ref = (a.double() @ w.double().T + b.double()).clamp_min(0)
    assert (out.double() - ref).abs().max().item() <= 2e-5          # exact products, fp32 accumulation order only
    out16 = ops.gemm_bias_act(a, w, b, relu=False, out_dtype=torch.bfloat16)
    ref16 = a.double() @ w.double().T + b.double()
    assert (out16.double() - ref16).abs().max().item() <= 2.0 ** -8 * ref16.abs().max().item() + 1e-5


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (1000, 256, 512), (4097, 1024, 96)])
def test_gemm_tf32_matches_fp64(dev, M, N, K):
    from pointnet_refine_b200 import ops
    g = torch.Generator(device=dev).manual_seed(M + N + K)
    a = torch.from_numpy(orc.round_tf32(torch.randn(M, K, generator=torch.Generator().manual_seed(1)).numpy())).to(dev)
    w = torch.from_numpy(orc.round_tf32((torch.randn(N, K, generator=torch.Generator().manual_seed(2)) / K ** 0.5).numpy())).to(dev)
    b = torch.randn(N, device=dev, generator=g)
    out = ops.gemm_bias_act(a, w, b, relu=False)
    ref = a.double() @ w.double().T + b.double()
    assert (out.double() - ref).abs().max().item() <= 2e-5          # operands already TF32-exact


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (1024, 2048, 2500), (64, 128, 30000), (512, 256, 4096)])
def test_gemm_tn_mn_major_operands(dev, M, N, K):
    """Weight-gradient shape: out = At^T Bt with both operands MN-major (K = points), split-K, ragged K."""
    from pointnet_refine_b200 import ops
    g = torch.Generator(device=dev).manual_seed(M + N + K)
    at = torch.randn(K, M, device=dev, generator=g).bfloat16()
    bt = (torch.randn(K, N, device=dev, generator=g) / K ** 0.5).bfloat16()
    out = ops.gemm_tn(at, bt)
    ref = at.double().T @ bt.double()
    assert (out.double() - ref).abs().max().item() <= 5e-5


# ------------------------------------------------------------------ encoder vs reference fixtures
@pytest.mark.parametrize("prec", list(TIERS))
@pytest.mark.parametrize("name", EVAL_CASES)
def test_encoder_matches_reference_golden(dev, name, prec):
    g, sd, ctx, line, (sc, sn) = load_case(name)
    m = _model(sd, dev, prec)
    with torch.no_grad():
        out = m.context_encoder.run_native(torch.from_numpy(ctx).to(dev), pool=True, argmax=True, fused=True, memory=True)
    gf, fused = out["global_feat"].cpu().numpy(), out["fused"].cpu().numpy()
    arg, mem = out["argmax"].cpu().numpy(), out["memory"].cpu().numpy()
    rng = max(1.0, float(np.abs(g["global_feat"]).max()))
    tol = TIERS[prec] * rng
    assert np.abs(gf - g["global_feat"]).max() <= tol
    assert np.abs(fused[:, ::sc, ::sn] - g["fused_sub"]).max() <= tol
    B, N = ctx.shape[:2]
    assert np.abs(fused.astype(np.float64).sum(2) - g["fused_csum"]).max() <= tol * N
    assert np.abs(fused.astype(np.float64).sum(1) - g["fused_psum"]).max() <= tol * 1024
    mrng = max(1.0, float(np.abs(g["memory_sub"]).max()))
    assert np.abs(mem[:, ::sn, ::sc] - g["memory_sub"]).max() <= TIERS[prec] * mrng
    # pooled outputs are consistent with the stored per-point map, exactly for max (same values reduced)
    assert np.array_equal(gf[:, :1024], fused.max(axis=2))
    np.testing.assert_allclose(gf[:, 1024:], fused.mean(axis=2, dtype=np.float64), rtol=0, atol=2e-6 * rng)
    assert np.array_equal(arg, fused.argmax(axis=2))                 # first index on ties, like torch.max
    safe = g["gap"] > 2 * tol                                        # reference argmax where it is unambiguous
    if safe.any():
        assert np.array_equal(arg[safe], g["argmax"][safe])
    untied = g["gap"] > 0                                            # every pair the reference decides without a tie
    rate = float((arg[untied] == g["argmax"][untied]).mean()) if untied.any() else 1.0
    report(test="encoder_golden", case=name, tier=prec, gf_err=float(np.abs(gf - g["global_feat"]).max()), range=rng,
           argmax_agreement_untied=rate, untied_pairs=int(untied.sum()), exact_subset_pairs=int(safe.sum()))
    if N >= 256:                                                     # (tiny segments: a handful of pairs, rate is noise)
        assert rate >= ARGMAX_FLOOR[prec], (name, prec, rate)


@pytest.mark.parametrize("prec", list(TIERS))
@pytest.mark.parametrize("name", EVAL_CASES)
def test_full_forward_matches_reference_golden(dev, name, prec):
    g, sd, ctx, line, _ = load_case(name)
    m = _model(sd, dev, prec)
    with torch.no_grad():
        out = m(torch.from_numpy(ctx).to(dev), torch.from_numpy(line).to(dev)).cpu().numpy()
    assert out.shape == g["out"].shape == (6, ctx.shape[0], 32, 3)
    err = float(np.abs(out - g["out"]).max())
    report(test="full_forward_golden", case=name, tier=prec, offsets_err=err, range=float(np.abs(g["out"]).max()))
    assert err <= _offset_tol(prec, g["out"]), (name, prec, err)


def test_module_encoder_interface(dev):
    """forward(x (B,4,N)) -> (global_feat, fused (B,1024,N)) like reference src/model.py:39-62."""
    g, sd, ctx, _, _ = load_case("b3_n1000_ragged")
    m = _model(sd, dev, "tf32")
    with torch.no_grad():
        gf, fused = m.context_encoder(torch.from_numpy(ctx).to(dev).transpose(2, 1))
    assert gf.shape == (3, 2048) and fused.shape == (3, 1024, 1000)
    assert (gf.cpu().numpy() - g["global_feat"]).__abs__().max() <= 1e-3 * max(1.0, np.abs(g["global_feat"]).max())


def test_heads_match_oracle(dev):
    from pointnet_refine_b200 import ops
    sd = synth.make_state_dict(3)
    rs = np.random.default_rng(5)
    for rows in (1, 31, 64, 1000):
        tgt = rs.standard_normal((rows, 256)).astype(np.float32)
        cur = rs.standard_normal((rows, 3)).astype(np.float32)
        noisy = rs.standard_normal((rows, 3)).astype(np.float32)
        t = {k: torch.from_numpy(v).to(dev) for k, v in sd.items() if k.startswith("reg_branches.2.")}
        cur_d = torch.from_numpy(cur).to(dev)
        cum = ops.head_forward(t["reg_branches.2.0.weight"], t["reg_branches.2.0.bias"], t["reg_branches.2.2.weight"],
                               t["reg_branches.2.2.bias"], torch.from_numpy(tgt).to(dev), cur_d,
                               torch.from_numpy(noisy).to(dev))
        delta = orc.head_forward(sd, 2, tgt, np.float64)
        np.testing.assert_allclose(cur_d.cpu().numpy(), cur + delta, rtol=0, atol=2e-5)
        np.testing.assert_allclose(cum.cpu().numpy(), cur + delta - noisy, rtol=0, atol=2e-5)


# ------------------------------------------------------------------ context side of the decoder (SURVEY.md 8f row 1)
@pytest.mark.parametrize("B,N,splits,ramp", [(1, 128, None, False), (2, 127, None, False), (3, 300, 1, False), (3, 300, 3, False),
                                             (1, 4096, None, False), (5, 1000, 2, True), (300, 3, None, False), (2, 65536, None, True)])
def test_ctx_attention_matches_fp64(dev, B, N, splits, ramp):
    """softmax(qfold kp^T) mem (lrn_ctx_attention) against fp64 on the same bf16 inputs; `ramp` makes the scores grow
    along the points so that the lazily rescaled running maximum is exercised; splits > 1 covers the merge."""
    from pointnet_refine_b200 import ops
    gen = torch.Generator(device=dev).manual_seed(B * 1000 + N)
    r = lambda *s: torch.randn(*s, device=dev, generator=gen)
    qf = (r(B, 256, 256) * (4.0 if ramp else 1.0) / 16).bfloat16()
    mem = r(B, N, 256).bfloat16()
    kp = mem.float() + 0.5 * r(B, N, 256)
    if ramp:
        kp = kp * torch.linspace(0.2, 3.0, N, device=dev)[None, :, None]
    kp = kp.bfloat16()
    out = ops.ctx_attention(qf, kp, mem, splits)
    ref = torch.softmax(qf.double() @ kp.double().transpose(1, 2) * np.log(2.0), dim=-1) @ mem.double()
    assert torch.isfinite(out).all()
    assert float((out.double() - ref).abs().max()) <= 1e-2 * max(1.0, float(ref.abs().max()))
    # strided views of a wider buffer (the layout LineRefineNet uses): same result, bit for bit
    wide = torch.empty(B, N, 512, dtype=torch.bfloat16, device=dev)
    wide[:, :, :256] = mem
    assert torch.equal(ops.ctx_attention(qf, kp, wide[:, :, :256], splits), out)
    # bf16 output: written by the kernel itself when the segment is not split, the fp32 result rounded once otherwise
    out16 = ops.ctx_attention(qf, kp, mem, splits, out_dtype=torch.bfloat16)
    assert out16.dtype == torch.bfloat16 and torch.equal(out16, out.bfloat16())


def test_pos_hidden_and_bf16_memory(dev):
    from pointnet_refine_b200 import ops
    g, sd, ctx, _, _ = load_case("b3_n1000_ragged")
    m = _model(sd, dev, "bf16")
    c = torch.from_numpy(ctx).to(dev)
    with torch.no_grad():
        mem32 = m.context_encoder.run_native(c, pool=False, memory=True)["memory"]
        memx = m.context_encoder.run_native(c, pool=False, memory=True, memory_bf16=True)["memory"]
        assert memx.shape == (3, 1000, 512) and memx.dtype == torch.bfloat16
        assert torch.equal(memx[:, :, :256], mem32.bfloat16())          # same accumulators, rounded once
        w1, b1 = m.pos_emb.mlp[0].weight, m.pos_emb.mlp[0].bias
        ops.pos_hidden(w1, b1, c, memx[:, :, 256:])
        ref = torch.relu(c[:, :, :3].double() @ w1.double().T + b1.double())
        assert float((memx[:, :, 256:].double() - ref).abs().max()) <= 2 ** -8 * max(1.0, float(ref.abs().max()))
        assert torch.equal(memx[:, :, :256], mem32.bfloat16())          # the memory half is left alone


def test_point_embed_tiled_layout_equals_row_major(dev):
    """Stand-alone first layer in the tiled operand layout of the default path == the row-major rows, re-tiled."""
    from pointnet_refine_b200 import ops
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "bf16")
    ctx = torch.from_numpy(synth.make_inputs(3, 1000, seed=2)[0]).to(dev)       # 3000 points: a ragged last tile
    folded = m.context_encoder.folded()
    rm = ops.point_embed(folded, ctx)                                            # (3000, 2048)
    tl = ops.point_embed(folded, ctx, tiled=True)                                # (24, 32, 128, 64)
    assert tl.shape == (24, 32, 128, 64)
    for blk, c0 in ((0, 0), (31, 1984)):
        flat = tl[:, blk].reshape(-1, 64)[:3000]
        assert torch.equal(flat, rm[:, c0:c0 + 64])


def test_query_side_kernels_match_torch(dev):
    """add + LayerNorm, the 32 x 32 self attention and the head update (SURVEY.md 8f row 2) against the stock modules."""
    import torch.nn.functional as F
    from pointnet_refine_b200 import ops
    gen = torch.Generator(device=dev).manual_seed(3)
    r = lambda *s: torch.randn(*s, device=dev, generator=gen)
    for B in (1, 7, 300):
        x, y = r(B, 32, 256) * 3 + 1, r(B, 32, 256)
        ln = torch.nn.LayerNorm(256).to(dev)
        with torch.no_grad():
            ln.weight.copy_(r(256)); ln.bias.copy_(r(256))
            assert float((ops.add_layernorm(x, y, ln) - ln(x + y)).abs().max()) <= 2e-5
            assert float((ops.add_layernorm(x, None, ln) - ln(x)).abs().max()) <= 2e-5
            mha = torch.nn.MultiheadAttention(256, 8, batch_first=True).to(dev).eval()
            q_in, v_in = r(B, 32, 256), r(B, 32, 256)
            ref = mha(q_in, q_in, value=v_in, need_weights=False)[0]
            W, bias = mha.in_proj_weight, mha.in_proj_bias
            qk = F.linear(q_in, W[:512], bias[:512])
            v = F.linear(v_in, W[512:], bias[512:])
            got = mha.out_proj(ops.self_attention32(qk, v))
            assert float((got - ref).abs().max()) <= 2e-5 * max(1.0, float(ref.abs().max()))
            hid, w2, b2 = r(B * 32, 128), r(3, 128), r(3)
            cur, noisy = r(B, 32, 3), r(B, 32, 3)
            want = cur + (hid.double() @ w2.double().T + b2.double()).view(B, 32, 3).float()
            cum = ops.head_update(hid, w2, b2, cur, noisy)
            assert float((cur - want).abs().max()) <= 1e-4 and float((cum - (want - noisy)).abs().max()) <= 1e-4


@pytest.mark.parametrize("M", [16, 32, 48])
@pytest.mark.parametrize("B,N", [(9, 300), (16, 1024)])
def test_full_forward_batched_vs_live_oracle(dev, B, N, M):
    """Every tier against the live oracle.  M = 32: the native decoder of the bf16 / tf32 tiers, B * 32 >= 256 query rows
    on the tcgen05 GEMMs (smaller batches use rows_linear); M = 16 / 48, and the fp32x3 tier: the stock fp32 decoder."""
    sd = synth.make_state_dict(21)
    ctx, line = synth.make_inputs(B, N, M=M, seed=5)
    ref = orc.line_refine_forward(sd, ctx, line)
    rng = max(1.0, float(np.abs(ref).max()))
    for prec in TIERS:
        m = _model(sd, dev, prec)
        with torch.no_grad():
            out = m(torch.from_numpy(ctx).to(dev), torch.from_numpy(line).to(dev))
        assert out.shape == (6, B, M, 3)
        err = float(np.abs(out.cpu().numpy() - ref).max())
        report(test="full_forward_live", B=B, N=N, M=M, tier=prec, offsets_err=err, range=rng)
        assert err <= _offset_tol(prec, ref), (prec, err)


def test_full_forward_chunking_and_segment_independence_at_scale(dev):
    """600 segments x 700 points: the decoder pass size (segments per pass, which also changes the attention kernel's
    split count) and the order of the segments must not matter beyond rounding; every segment is independent."""
    sd = synth.make_state_dict(4)
    m = _model(sd, dev, "bf16")
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(600, 700, seed=31))
    with torch.no_grad():
        full = m(ctx, line)
        m.segment_chunk = 5                               # 40 segments per pass on the attention path
        small = m(ctx, line)
        m.segment_chunk = 256
        perm = torch.randperm(600, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
        shuffled = m(ctx[perm], line[perm])
        alone = m(ctx[17:18], line[17:18])                # B = 1: stock-op query side, attention split over clusters
    rng = max(1.0, float(full.abs().max()))
    assert torch.isfinite(full).all()
    assert float((small - full).abs().max()) <= 5e-3 * rng
    assert float((shuffled - full[:, perm]).abs().max()) <= 5e-3 * rng
    assert float((alone[:, 0] - full[:, 17]).abs().max()) <= 5e-3 * rng


# ------------------------------------------------------------------ live oracle, odd shapes
@pytest.mark.parametrize("B,N", [(1, 127), (1, 129), (7, 300), (4, 4096), (300, 3)])
def test_encoder_vs_live_oracle(dev, B, N):
    sd = synth.make_state_dict(11)
    ctx, _ = synth.make_inputs(B, N, seed=77)
    gf_o, fused_o, _ = orc.encoder_forward(sd, ctx)
    rng = max(1.0, float(np.abs(gf_o).max()))
    for prec, t in TIERS.items():
        m = _model(sd, dev, prec)
        with torch.no_grad():
            out = m.context_encoder.run_native(torch.from_numpy(ctx).to(dev), pool=True, fused=True)
        assert np.abs(out["global_feat"].cpu().numpy() - gf_o).max() <= t * rng
        assert np.abs(out["fused"].cpu().numpy() - fused_o.transpose(0, 2, 1)).max() <= t * rng


# ------------------------------------------------------------------ size-independent properties at scale
def test_properties_at_scale(dev):
    """Chunk invariance, permutation invariance within a segment, segment independence and
    determinism of the max-pool at BASELINE.json's full configs[1] size (4096 x 4096 points)."""
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "bf16")
    B, N = 4096, 4096                     # BASELINE.json configs[1], full size
    ctx = torch.randn(B, N, 4, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    enc = m.context_encoder
    with torch.no_grad():
        base = enc.run_native(ctx, pool=True, argmax=True)
        enc.chunk_rows = 128 * 37 * 5                                  # waves that cut through segments
        chunked = enc.run_native(ctx, pool=True, argmax=True)
        enc.chunk_rows = 0
        perm = torch.randperm(N, device=dev)
        permuted = enc.run_native(ctx[:, perm].contiguous(), pool=True)
        rev = enc.run_native(ctx.flip(0).contiguous(), pool=True)
    gf = base["global_feat"]
    assert torch.isfinite(gf).all() and (gf >= 0).all()
    assert torch.equal(gf[:, :1024], chunked["global_feat"][:, :1024])           # max is order independent
    assert torch.equal(base["argmax"], chunked["argmax"])
    assert (gf[:, 1024:] - chunked["global_feat"][:, 1024:]).abs().max() <= 1e-5
    assert torch.equal(gf[:, :1024], permuted["global_feat"][:, :1024])
    assert (gf[:, 1024:] - permuted["global_feat"][:, 1024:]).abs().max() <= 1e-5
    assert torch.equal(gf[:, :1024], rev["global_feat"].flip(0)[:, :1024])       # segments are independent
    assert (gf[:, :1024] >= gf[:, 1024:]).all()                                  # max >= mean
    # spot-check 2 segments against the oracle
    o = orc.encoder_forward(sd, ctx[:2].cpu().numpy())[0]
    assert np.abs(gf[:2].cpu().numpy() - o).max() <= 1e-2 * max(1.0, np.abs(o).max())


def test_large_context_stress(dev):
    """BASELINE.json configs[4] shape class: very long segments reduce across many tiles and waves."""
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "bf16")
    B, N = 4, 65536
    ctx = torch.randn(B, N, 4, device=dev, generator=torch.Generator(device=dev).manual_seed(6))
    with torch.no_grad():
        a = m.context_encoder.run_native(ctx, pool=True, argmax=True)
        dup = m.context_encoder.run_native(torch.cat([ctx, ctx], dim=1), pool=True, argmax=True)
    # duplicating every point leaves max, mean and (first-index) argmax unchanged
    assert torch.equal(a["global_feat"][:, :1024], dup["global_feat"][:, :1024])
    assert torch.equal(a["argmax"], dup["argmax"])
    assert (a["global_feat"][:, 1024:] - dup["global_feat"][:, 1024:]).abs().max() <= 1e-5
    o = orc.encoder_forward(sd, ctx[:1, :].cpu().numpy())[0]
    assert np.abs(a["global_feat"][:1].cpu().numpy() - o).max() <= 1e-2 * max(1.0, np.abs(o).max())


# ------------------------------------------------------------------ error behaviour
def test_errors_are_loud(dev):
    from pointnet_refine_b200 import _lib, ops
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "bf16")
    with pytest.raises(ValueError):
        m.context_encoder.run_native(torch.zeros(0, 16, 4, device=dev))
    with pytest.raises(ValueError):
        m.context_encoder.run_native(torch.zeros(2, 16, 3, device=dev))
    folded = m.context_encoder.folded()
    st = _lib.lib.lrn_encoder_forward(folded.blob.data_ptr(), 0, None, 1, 16, 1, None, None, None, None, 0, None, 0, None)
    assert st == 6 and b"null" in _lib.lib.lrn_last_error()
    st = _lib.lib.lrn_encoder_forward(folded.blob.data_ptr(), 0, folded.blob.data_ptr(), 0, 16, 1, None, None, None, None,
                                      0, folded.blob.data_ptr(), 0, None)
    assert st == 1                                                   # empty input -> LRN_ERR_BAD_SHAPE
    with pytest.raises(TypeError):
        ops.gemm_bias_act(torch.zeros(8, 64, device=dev), torch.zeros(128, 64, device=dev).bfloat16(), None)
    # decoder context side / scene front end: wrong types, shapes and parameters are refused, not worked around
    bf = lambda *s: torch.zeros(*s, device=dev, dtype=torch.bfloat16)
    with pytest.raises(TypeError):
        ops.ctx_attention(torch.zeros(1, 256, 256, device=dev), bf(1, 64, 256), bf(1, 64, 256))
    with pytest.raises(ValueError):
        ops.ctx_attention(bf(1, 128, 256), bf(1, 64, 256), bf(1, 64, 256))
    with pytest.raises(RuntimeError):
        ops.ctx_attention(bf(1, 256, 256), bf(1, 64, 256), bf(1, 64, 256), splits=5)          # more splits than point tiles
    with pytest.raises(RuntimeError):
        m.precision = "tf32"
        try:
            m.context_encoder.run_native(torch.zeros(1, 16, 4, device=dev), pool=False, memory=True, memory_bf16=True)
        finally:
            m.precision = "bf16"
    from pointnet_refine_b200 import scene as sc
    pts = torch.zeros(100, 4, device=dev)
    line = [[0.0, 0.0, 0.0], [1.0, 0.0, 0.0]]
    with pytest.raises(TypeError):
        sc.build_segments(pts.cpu(), [line])
    with pytest.raises(ValueError):
        sc.build_segments(pts, [])
    with pytest.raises(RuntimeError):
        sc.build_segments(pts, [line], num_context_points=5000)                                  # N <= 4096
    with pytest.raises(RuntimeError):
        sc.build_segments(pts, [line], crop_radius=100.0, decay_scale=1.0)                       # weights would underflow


def test_refold_after_parameter_update(dev):
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "tf32")
    ctx = torch.from_numpy(synth.make_inputs(2, 256, seed=3)[0]).to(dev)
    with torch.no_grad():
        a = m.context_encoder.run_native(ctx, pool=True)["global_feat"].clone()
        m.context_encoder.bn5.running_mean.add_(0.05)                # e.g. a training step / checkpoint load
        b = m.context_encoder.run_native(ctx, pool=True)["global_feat"]
    sd2 = dict(sd)
    sd2["context_encoder.bn5.running_mean"] = sd["context_encoder.bn5.running_mean"] + np.float32(0.05)
    o = orc.encoder_forward(sd2, ctx.cpu().numpy())[0]
    assert not torch.equal(a, b)
    assert np.abs(b.cpu().numpy() - o).max() <= 1e-3 * max(1.0, np.abs(o).max())


def test_invalidate_after_data_edit(dev):
    """In-place edits through `.data` do not bump `_version`: the caches keep the old weights until invalidate()."""
    sd = synth.make_state_dict(5)
    m = _model(sd, dev, "bf16")
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(2, 300, seed=8))
    with torch.no_grad():
        a = m(ctx, line).clone()
        for p in m.parameters():
            p.data.mul_(1.01)
        m.invalidate()
        b = m(ctx, line)
        m2 = _model({k: (v * 1.01 if v.dtype.kind == "f" and not k.endswith(("running_mean", "running_var")) else v) for k, v in sd.items()},
                    dev, "bf16")
        c = m2(ctx, line)
    assert float((a - b).abs().max()) > 0
    assert torch.equal(b, c)


def test_host_pipeline_matches_direct_call(dev):
    """Chunked, copy/compute-overlapped host streaming returns exactly what one direct call returns."""
    from pointnet_refine_b200.stream import HostEncoderPipeline
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, "bf16")
    host = torch.randn(700, 256, 4, generator=torch.Generator().manual_seed(9)).pin_memory()
    with torch.no_grad():
        direct = m.context_encoder.run_native(host.to(dev), pool=True)["global_feat"].cpu()
    got = HostEncoderPipeline(m.context_encoder, segments_per_chunk=128).global_feat(host)
    assert torch.equal(got[:, :1024], direct[:, :1024])
    assert (got[:, 1024:] - direct[:, 1024:]).abs().max() <= 1e-5


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
@pytest.mark.parametrize("B,N", [(1, 1024), (24, 512)])
def test_cuda_graph_replay_is_bit_identical(dev, B, N, prec):
    """B = 1 whole-scene style call (inference_whole_scene.py:130-139) and a batch large enough for the native query side:
    one graph replay == the eager launches, also after invalidate() and an eager call have rebuilt every prepared weight
    (the graph reads the ones it was captured with, which it keeps alive)."""
    import pointnet_refine_b200 as prb
    sd = synth.make_state_dict(0)
    m = _model(sd, dev, prec)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(B, N, seed=21))
    with torch.no_grad():
        eager = m(ctx, line).clone()
        runner = prb.GraphedLineRefineNet(m, B, N)
        m.invalidate()
        m(ctx, line)
        for _ in range(3):
            out = runner(ctx, line)
        torch.cuda.synchronize()
    assert torch.equal(out, eager)


def test_compat_shim_runs_reference_smoke(dev):
    """The body of the reference's own smoke test (src/model.py:236-246: default-constructed model, randn(2,1024,4) /
    randn(2,32,3), expects (6,2,32,3) and prints the parameter count) through `from src.model import LineRefineNet` with
    <repo>/compat first on sys.path -- on the GPU, in the module's default train mode and in eval mode -- plus the
    checkpoint round trip of inference_whole_scene.py:202-204."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r"""
import os, sys, tempfile
root = sys.argv[1]
sys.path[:0] = [os.path.join(root, "compat"), root]
import torch
from src.model import LineRefineNet
device = torch.device("cuda")
model = LineRefineNet().to(device)
ctx = torch.randn(2, 1024, 4, device=device)
line = torch.randn(2, 32, 3, device=device)
out = model(ctx, line)                                     # train mode, like `python src/model.py`
print(out.shape)
assert tuple(out.shape) == (6, 2, 32, 3) and torch.isfinite(out).all()
print(f"Model Parameters: {sum(p.numel() for p in model.parameters())}")
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "best_model.pth")
    torch.save(model.state_dict(), path)
    m2 = LineRefineNet().to(device)
    m2.load_state_dict(torch.load(path, map_location=device))
m2.eval()
model.eval()
with torch.no_grad():
    a = model(ctx, line)[-1]                               # inference_whole_scene.py:137-139
    b = m2(ctx, line)[-1]
assert tuple(a.shape) == (2, 32, 3) and torch.equal(a, b)
print("compat smoke ok")
"""
    r = subprocess.run([sys.executable, "-c", code, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "compat smoke ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
    assert "Model Parameters: 9695954" in r.stdout
