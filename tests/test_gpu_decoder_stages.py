"""The eval decoder (`LineRefineNet._refine_native`, bf16 and tf32 tiers) checked stage by stage on its own intermediates,
against fp64 references of the same arithmetic.

The end-to-end tests allow 1e-2 of the range (bf16) or 1e-3 (tf32) on the offsets, which a decoder kernel or weight fold
that is subtly wrong still passes.  Here a real forward is recorded at the `ops` entry points it calls (every tensor
argument cloned before the call, results and in-place targets after it) and every recorded call is checked on the inputs
it actually received, together with the chain: each stage's activation input is, bit for bit, the recorded output of the
stage that `DetrTransformerDecoderLayer.forward` says feeds it.  The prepared weights are checked against the state
dict in fp64, and the two attention kernels and the split merge are driven directly at the edges where they go wrong.

Bounds (u = 2^-24, the fp32 unit roundoff; S = sum |a * b| + |bias| in fp64; first-order error analysis):
  * rows_linear: each of the eight warps runs one FMA chain over K/8 terms, the block adds bias + 8 partials in order:
    (K/8 + 9) u S.  `add=`: the operand is the fp32 sum (one rounding), mirrored exactly.  `mlp3=`: every hidden unit is a
    3-FMA chain, off by e_k = 4 u (|b1_k| + sum |w1 c|), propagated as sum_k |w_nk| e_k.  bf16 output: + 2^-8 (|ref| + acc).
  * tcgen05 GEMMs (as in test_gpu_encoder_stages): (steps + 2) 2^-23 S, steps = K/8 (TF32 kind) or K/16 (bf16 kind), plus
    half an output ulp (2^-8 relative for bf16).  tf32 tier: both operands TF32-exact, equal to the nearest TF32 value of
    the fp32 input.  bf16 tier with fp32 operands: the tensor core truncates each operand to TF32 (DESIGN.md section 3b);
    the mirror truncates too, and the fraction stored bit-exact is reported.
  * pos_hidden / query_pos_hidden: 3-FMA chain, 4 u S; then bf16 (2^-8) or TF32 rounding (2^-11, and TF32-exact).
    add: bit-exact, with the TF32 rounding where asked.
  * self_attention32: score s_j = (q / sqrt 32) . k_j from 4 chains of 8 FMAs + 2 adds and the rounded scale: 12 u T_j
    (T_j = sum |q k_j| / sqrt 32).  Each weight exp(s_j - m) is then off by eps_j = 12 u T_j + u (m - s_j) + 2^-22 (the
    subtraction and expf's 2 ulp) relative; normalising moves every weight by at most sum_j P_j eps_j; the 31 adds of the
    sum, the reciprocal, the product and the 32-term output FMA chain add 66 u.  Bound per output: sum_j P_j |v_j| eps_j
    + (sum_j P_j eps_j + 66 u) sum_j P_j |v_j|.
  * cross_attention32: as above with 2 chains of 16 FMAs (19 u T_j) and __expf = ex2.approx(x log2 e): 2 u |x| + 2^-22 per
    factor; a weight goes through its own exponential, the running rescales and the merge factor, whose arguments add up
    to at most (m - s_j) + 2 R (R = the row's score range), and (nb + 1) approximations (nb = key blocks per warp).  The
    accumulators see n_w = 32 nb FMAs and nb rescales, the merge 8 + 8 FMAs and one division.
  * add_layernorm: z = x + y in fp32 (mirrored exactly); the mean from 8 in-thread adds + 5 shuffle levels (13 u sum|z|);
    the variance likewise plus the squares (17 u sum a^2 + 2 d_mean sum |a|); rsqrtf 2 ulp (2^-22); the final
    a * rstd * gamma + beta three roundings.
  * ctx_attention (bf16): scores from exact bf16 products with fp32 accumulation over 16 MMA steps (18 2^-23 T, log2
    units); p = ex2.approx(S - m_ref): ln2 (dS + u (m - S + 8)) + 2^-22 relative (m_ref trails the maximum by at most 8);
    P enters O rounded to bf16 (2^-8 relative, scale-free, so the lazily moved m_ref does not enter) while l sums the
    unrounded fp32 p: (20 + 2 steps) u; O accumulates over 8 MMA steps per 128 points: (8 steps + 2) 2^-23.  lse =
    m_ref + log2f(l): sum_j P_j dS_j + (relative error of l) / ln2 + 2 u |log2 l| + u |lse|.  The merge weights
    2^(lse_s - max) / sum: ln2 (d lse_s + max d lse) + 2^-22 (exp2f) + ln2 u |lse_s - max| + (S + 2) u, and S FMAs.
  * head_update: 4 in-thread terms + 5 shuffle levels + bias + the add to `current`: 11 u (S + |b2|) + u |result|; the
    cumulative offset is the fp32 difference of the updated `current` and the noisy line, bit for bit.
The worst error / bound of every check is reported (parity_report.jsonl).
"""
import math

import numpy as np
import pytest
import torch

from oracle import synth
from tests.golden_util import report
from tests.test_gpu_encoder_stages import TINY, _bits, _check_linear, _rna_tf32, dev  # noqa: F401  (dev: fixture)

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
LN2 = math.log(2.0)
D = 256
ENTRY_POINTS = ("encoder_forward", "rows_linear", "gemm_bias_act", "query_pos_hidden", "add", "pos_hidden",
                "self_attention32", "add_layernorm", "ctx_attention", "cross_attention32", "head_update")
IN_PLACE = {"head_update": 3, "pos_hidden": 3}          # argument written by the call (current; memx[:, :, 256:])


# ------------------------------------------------------------------ small helpers
def _same(a, b, what):
    """Bit equality of two tensors (any shapes with the same elements in row-major order), or both None."""
    if a is None or b is None:
        assert a is None and b is None, what
        return
    assert a.dtype == b.dtype and a.numel() == b.numel(), (what, a.dtype, b.dtype, tuple(a.shape), tuple(b.shape))
    assert torch.equal(_bits(a.reshape(-1)), _bits(b.reshape(-1))), what


def _tf32_exact(t, what):
    assert int((_bits(t) & 0x1FFF).abs().max()) == 0, f"{what}: not TF32-exact"


def _trunc_tf32(t):
    """fp32 -> TF32 by dropping the low 13 mantissa bits (what the tensor core does to an fp32 operand)."""
    return (t.contiguous().view(torch.int32) & -0x2000).view(torch.float32)


def _ratio(got, want, bound):
    return float(((got.double() - want).abs() / (bound + TINY)).nan_to_num(nan=math.inf).max())


def _clone(v):
    if isinstance(v, torch.Tensor):
        return v.detach().clone()
    if isinstance(v, (tuple, list)):
        return type(v)(_clone(x) for x in v)
    if isinstance(v, dict):
        return {k: _clone(x) for k, x in v.items()}
    return v


class Stages:
    """Worst error / bound per stage of one case; every check asserts and the worst ratios are reported."""

    def __init__(self, case, tier):
        self.case, self.tier, self.worst = case, tier, {}

    def check(self, stage, ratio, exact=None):
        r, e = self.worst.get(stage, (0.0, None))
        self.worst[stage] = (max(r, ratio), exact if e is None else (min(e, exact) if exact is not None else e))
        if ratio > 1.0:
            report(test="decoder_stages", case=self.case, tier=self.tier, stage=stage, ratio=ratio, failed=True)
        assert ratio <= 1.0, f"{self.case} {self.tier} {stage}: error / bound = {ratio:.3g}"

    def flush(self):
        for stage, (ratio, exact) in self.worst.items():
            report(test="decoder_stages", case=self.case, tier=self.tier, stage=stage, ratio=ratio, exact=exact)


# ------------------------------------------------------------------ stage mirrors
def _fma3(w1, b1, c):
    """relu(c[:, :3] @ w1.T + b1) in fp64 and the error of its 3-FMA chain in fp32."""
    c, w1, b1 = c.reshape(-1, c.shape[-1])[:, :3].double(), w1.double(), b1.double()
    ref = torch.addmm(b1, c, w1.T)
    return ref.clamp_min(0), 4 * U * torch.addmm(b1.abs(), c.abs(), w1.abs().T)


def _check_rows_linear(r, st, stage):
    x, w, b = r.args[:3]
    add, mlp3 = r.kw.get("add"), r.kw.get("mlp3")
    relu, bf16_out = r.kw.get("relu", False), r.kw.get("out_dtype", torch.float32) == torch.bfloat16
    K = w.shape[1]
    w64, b64 = w.double(), b.double()
    if mlp3 is not None:
        h, e = _fma3(mlp3[0], mlp3[1], x)
        extra = e @ w64.abs().T
    else:
        h = (x if add is None else x + add).reshape(-1, K).double()
        extra = 0.0
    ref = torch.addmm(b64, h, w64.T)
    acc = (K // 8 + 9) * U * torch.addmm(b64.abs(), h.abs(), w64.abs().T) + extra
    want = ref.clamp_min(0) if relu else ref
    bound = acc + (2.0 ** -8 * (ref.abs() + acc) if bf16_out else 0.0)
    st.check(stage, _ratio(r.out.reshape(ref.shape), want, bound))


def _check_gemm(g, mode, st, stage):
    """mode: 'tf32' (TF32-exact fp32 operands), 'trunc' (fp32 operands the tensor core truncates), 'bf16'."""
    a, w, b = g.args[:3]
    relu, out_dtype = g.kw.get("relu", False), g.kw.get("out_dtype")
    bf16_out = out_dtype == torch.bfloat16 or (out_dtype is None and a.dtype == torch.bfloat16)
    K = a.shape[1]
    if mode == "tf32":
        _tf32_exact(a, stage)
        _tf32_exact(w, stage)
    steps = K // 16 if mode == "bf16" else K // 8
    u = 2.0 ** -8 if bf16_out else 0.0
    rounding = (lambda v: v.float().bfloat16().double()) if bf16_out else None
    got = g.out.double()
    if mode == "trunc":   # report how the nearest-TF32 reading would fare, then assert the truncating one
        x, ww = _rna_tf32(a).double(), _rna_tf32(w).double()
        ref = torch.addmm(b.double(), x, ww.T)
        ref = ref.clamp_min(0) if relu else ref
        acc = (steps + 2) * 2.0 ** -23 * torch.addmm(b.double().abs(), x.abs(), ww.abs().T)
        report(test="decoder_stages", case=st.case, tier=st.tier, stage=stage + " (nearest-TF32 mirror)",
               ratio=_ratio(got, ref, acc + u * (ref.abs() + acc)))
        a, w = _trunc_tf32(a), _trunc_tf32(w)
    ratio, exact = _check_linear(a.double(), w.double(), b.double(), got, steps=steps, u=u, relu=relu, rounding=rounding,
                                 what=f"{st.case} {st.tier} {stage}")
    st.check(stage, ratio, exact)


def _check_add(a, st, stage):
    x, y = a.args[0], a.args[1] if len(a.args) > 1 else a.kw.get("b")
    want = x if y is None else x + y
    if a.kw.get("round_tf32", False):
        want = _rna_tf32(want)
    _same(a.out, want, f"{st.case} {st.tier} {stage}")
    st.check(stage, 0.0)


def _check_query_pos_hidden(q, st, stage):
    w1, b1, coords = q.args[:3]
    rnd = q.kw.get("round_tf32", False)
    ref, e = _fma3(w1, b1, coords)
    got = q.out.reshape(ref.shape)
    bound = e
    if rnd:
        _tf32_exact(got, stage)
        bound = e + 2.0 ** -11 * (ref.abs() + e)
    st.check(stage, _ratio(got, ref, bound))


def _check_pos_hidden(p, st, stage):
    w1, b1, ctx = p.args[:3]
    ref, e = _fma3(w1, b1, ctx)
    got = p.after.reshape(ref.shape)
    st.check(stage, _ratio(got, ref, e + 2.0 ** -8 * (ref.abs() + e)))


def _attn32_mirror(q, k, v, cross):
    """fp64 attention of 32 queries per segment, 8 heads x 32, and the bound of the fp32 kernel (module docstring).
    q (B, 32, 256), k / v (B, N, 256) -> ref, bound (B, 32, 256)."""
    B, N = k.shape[:2]
    heads = lambda t: t.reshape(B, -1, 8, 32).transpose(1, 2).double()
    qh, kh, vh = heads(q), heads(k), heads(v)
    S = qh @ kh.transpose(-1, -2) / math.sqrt(32)
    T = qh.abs() @ kh.abs().transpose(-1, -2) / math.sqrt(32)
    M = S.amax(-1, keepdim=True)
    P = torch.softmax(S, -1)
    if cross:
        nb = (N + 255) // 256
        R = M - S.amin(-1, keepdim=True)
        eps = 19 * U * T + 2 * U * ((M - S) + 2 * R) + (nb + 1) * 2.0 ** -22
        tail = (2 * 32 * nb + 3 * nb + 29) * U
    else:
        eps = 12 * U * T + U * (M - S) + 2.0 ** -22
        tail = 66 * U
    A0 = P @ vh.abs()
    bound = (P * eps) @ vh.abs() + ((P * eps).sum(-1, keepdim=True) + tail) * A0
    back = lambda t: t.transpose(1, 2).reshape(B, 32, 256)
    return back(P @ vh), back(bound)


def _check_layernorm(n, st, stage):
    x, y, norm = n.args[:3]
    z = (x if y is None else x + y).reshape(-1, D).double()
    g, beta, eps = norm.weight.detach().double(), norm.bias.detach().double(), float(norm.eps)
    mu = z.mean(-1, keepdim=True)
    a = z - mu
    var = (a * a).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    ref = a * rstd * g + beta
    dmu = 13 * U * z.abs().sum(-1, keepdim=True) / D + U * mu.abs()
    da = dmu + U * (a.abs() + dmu)
    dq = 17 * U * (a * a).sum(-1, keepdim=True) + 2 * dmu * a.abs().sum(-1, keepdim=True)
    dvar = dq / D + U * (var + eps)
    rel = 0.5 * dvar / (var + eps) + 2.0 ** -22 + U
    bound = g.abs() * rstd * (da + a.abs() * (rel + 2 * U)) + U * ref.abs()
    st.check(stage, _ratio(n.out.reshape(ref.shape), ref, bound))


def _ctx_mirror(qf, kp, mem, splits):
    """fp64 softmax_2(qf kp^T) mem per split and merged, with the kernel's bounds (module docstring).  Returns
    ([(part ref, part bound, lse ref, lse bound)] per split, merged ref, merged bound)."""
    B, N, _ = kp.shape
    total = (N + 127) // 128
    per = (total + splits - 1) // splits
    q = qf.double()
    parts, A0s = [], []
    for s in range(splits):
        a, e = s * per * 128, min(N, (s + 1) * per * 128)
        k, v = kp[:, a:e].double(), mem[:, a:e].double()
        steps = (e - a + 127) // 128
        S = q @ k.transpose(1, 2)
        dS = 18 * 2.0 ** -23 * (q.abs() @ k.abs().transpose(1, 2))
        m = S.amax(-1, keepdim=True)
        E = torch.exp2(S - m)
        l = E.sum(-1, keepdim=True)
        P = E / l
        e_exp = LN2 * U * (m - S + 8) + 2.0 ** -22
        eps = LN2 * dS + e_exp
        A0 = P @ v.abs()
        lrel = (20 + 2 * steps) * U
        bound = (P * eps) @ v.abs() + 2.0 ** -8 * A0 + ((P * eps).sum(-1, keepdim=True) + lrel + 2 * U
                                                        + (8 * steps + 2) * 2.0 ** -23) * A0
        lse = m + torch.log2(l)
        dlse = (P * dS).sum(-1, keepdim=True) + ((P * e_exp).sum(-1, keepdim=True) + lrel) / LN2 \
            + 2 * U * torch.log2(l).abs() + U * lse.abs()
        parts.append((P @ v, bound, lse[..., 0], dlse[..., 0]))
        A0s.append(A0)
    if splits == 1:
        return parts, parts[0][0], parts[0][1]
    L = torch.stack([p[2] for p in parts], 1)          # (B, S, 256)
    dL = torch.stack([p[3] for p in parts], 1)
    mx = L.amax(1, keepdim=True)
    w = torch.exp2(L - mx)
    w = w / w.sum(1, keepdim=True)
    werr = LN2 * (dL + dL.amax(1, keepdim=True)) + 2.0 ** -22 + LN2 * U * (L - mx).abs() + (splits + 2) * U
    ref = sum(w[:, s, :, None] * parts[s][0] for s in range(splits))
    bound = sum(w[:, s, :, None] * (parts[s][1] + (werr[:, s, :, None] + splits * U) * A0s[s]) for s in range(splits))
    return parts, ref, bound


def _ctx_splits(B, N):
    from pointnet_refine_b200._lib import lib
    return lib.lrn_ctx_attention_splits(B, N)


def _check_ctx(c, st, stage):
    qf, kp, mem = c.args[:3]
    splits = c.kw.get("splits") or (c.args[3] if len(c.args) > 3 and c.args[3] else _ctx_splits(kp.shape[0], kp.shape[1]))
    _, ref, bound = _ctx_mirror(qf, kp, mem, splits)
    if c.kw.get("out_dtype", torch.float32) == torch.bfloat16:
        bound = bound + 2.0 ** -8 * (ref.abs() + bound)
    else:
        bound = bound + U * ref.abs()
    st.check(stage, _ratio(c.out, ref, bound))


def _check_head_update(h, st, stage):
    hid, w2, b2, cur, noisy = h.args[:5]
    w64, b64 = w2.double(), b2.double()
    hv = hid.reshape(-1, 128).double()
    d = torch.addmm(b64, hv, w64.T)
    S = torch.addmm(b64.abs(), hv.abs(), w64.abs().T)
    ref = cur.reshape(-1, 3).double() + d
    new = h.after.reshape(-1, 3)
    st.check(stage, _ratio(new, ref, 11 * U * S + U * ref.abs() + 12 * U * U * S))
    _same(h.out, new - noisy.reshape(-1, 3), f"{st.case} {st.tier} {stage}: cumulative offset")


# ------------------------------------------------------------------ recording harness
class Call:
    def __init__(self, name, args, kw):
        self.name, self.args, self.kw = name, args, kw
        self.out = self.after = None


@pytest.fixture
def record(monkeypatch):
    """record(model, ctx, line) -> (output, [Call]): an eval forward with every ops entry point the decoder uses wrapped;
    arguments are cloned before the call, the result (and the in-place target) after it."""
    from pointnet_refine_b200 import ops

    def run(m, ctx, line):
        calls = []
        for name in ENTRY_POINTS:
            orig = getattr(ops, name)

            def wrapped(*args, _orig=orig, _name=name, **kw):
                c = Call(_name, _clone(args), _clone(kw))
                res = _orig(*args, **kw)
                c.out = _clone(res)
                if _name in IN_PLACE:
                    c.after = _clone(args[IN_PLACE[_name]])
                calls.append(c)
                return res
            monkeypatch.setattr(ops, name, wrapped)
        try:
            with torch.no_grad():
                out = m(ctx, line)
            torch.cuda.synchronize()
        finally:
            monkeypatch.undo()
        return out, calls
    return run


def _model(prec, dev, seed=13):
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to(dev).eval()
    m.load_state_dict(synth.to_torch(synth.make_state_dict(seed)), strict=True)
    m.precision = prec
    return m


def _walk(calls, m, prec, ctx, line, out, st):
    """Check every recorded call in the order _refine_native issues them: the chain (inputs = outputs of the stage that
    feeds them) and the stage itself."""
    it = iter(calls)

    def take(name):
        c = next(it, None)
        assert c is not None and c.name == name, f"{st.case} {prec}: expected {name}, got {c and c.name}"
        return c

    tf32 = prec == "tf32"
    B, N = ctx.shape[:2]
    from pointnet_refine_b200.ops import DEFAULT_CHUNK_ROWS
    chunk = (max(1, min(8 * m.segment_chunk, (4 * DEFAULT_CHUNK_ROWS) // N)) if not tf32
             else max(1, min(m.segment_chunk, (1 << 20) // N)))
    pe0, pe2 = m.pos_emb.mlp[0], m.pos_emb.mlp[2]
    for s0 in range(0, B, chunk):
        cx, ln = ctx[s0:s0 + chunk], line[s0:s0 + chunk]
        Bc = cx.shape[0]
        big = Bc * 32 >= 256

        def lin(x, w, b, relu=False, out_dtype=None, add=None, what=""):
            w, b = w.detach(), b.detach()
            if not big:
                r = take("rows_linear")
                _same(r.args[0], x, f"{what} input")
                _same(r.args[1], w, f"{what} weight")
                _same(r.kw.get("add"), add, f"{what} addend")
                assert r.kw.get("relu", False) == relu and r.kw.get("out_dtype", torch.float32) == (out_dtype or torch.float32)
                _check_rows_linear(r, st, "rows_linear")
                return r.out
            if tf32:
                a = take("add")
                _same(a.args[0], x, f"{what} input")
                _same(a.args[1], add, f"{what} addend")
                assert a.kw.get("round_tf32"), f"{what}: the operand must be rounded to the nearest TF32 value"
                _check_add(a, st, "add (round_tf32)")
                x = a.out
            elif add is not None:
                a = take("add")
                _same(a.args[0], x, f"{what} input")
                _same(a.args[1], add, f"{what} addend")
                _check_add(a, st, "add")
                x = a.out
            g = take("gemm_bias_act")
            _same(g.args[0], x, f"{what} operand")
            _same(g.args[1], _rna_tf32(w) if tf32 else w, f"{what} weight operand")
            _same(g.args[2], b, f"{what} bias")
            _check_gemm(g, "tf32" if tf32 else "trunc", st,
                        "gemm tf32" if tf32 else ("gemm fp32 operands, bf16 out" if out_dtype == torch.bfloat16
                                                  else "gemm fp32 operands"))
            return g.out.view(Bc, -1, w.shape[0])

        e = take("encoder_forward")
        _same(e.args[1], cx, "encoder input")
        memory = e.out["memory"]
        if tf32:
            wk, bk, wv, bv, w2 = m._kv_weights()
            q = take("query_pos_hidden")
            _same(q.args[2], cx, "context pos hidden input")
            _check_query_pos_hidden(q, st, "query_pos_hidden (round_tf32)")
            g = take("gemm_bias_act")
            _same(g.args[0], q.out, "pos_emb layer 2 operand")
            _same(g.args[1], _rna_tf32(pe2.weight.detach()), "pos_emb layer 2 weight")
            _check_gemm(g, "tf32", st, "gemm tf32 (context)")
            a = take("add")
            _same(a.args[0], memory, "K operand: memory")
            _same(a.args[1], g.out, "K operand: pos")
            assert a.kw.get("round_tf32"), "K operand must be rounded to the nearest TF32 value"
            _check_add(a, st, "add (round_tf32)")
            gk = take("gemm_bias_act")
            _same(gk.args[0], a.out, "K projection operand")
            _same(gk.args[1], wk, "K weights")
            _check_gemm(gk, "tf32", st, "gemm tf32 (context)")
            a = take("add")
            _same(a.args[0], memory, "V operand: memory")
            assert a.args[1] is None and a.kw.get("round_tf32"), "V operand must be rounded to the nearest TF32 value"
            _check_add(a, st, "add (round_tf32)")
            gv = take("gemm_bias_act")
            _same(gv.args[0], a.out, "V projection operand")
            _same(gv.args[1], wv, "V weights")
            _check_gemm(gv, "tf32", st, "gemm tf32 (context)")
            k_all, v_all = gk.out.view(Bc, N, 6 * D), gv.out.view(Bc, N, 6 * D)
        else:
            layers_w, wx, b2 = m._attn_weights()
            p = take("pos_hidden")
            _same(p.args[2], cx, "pos_hidden input")
            _check_pos_hidden(p, st, "pos_hidden")
            memx = memory.clone()
            memx[:, :, D:] = p.after
            g = take("gemm_bias_act")
            _same(g.args[0], memx, "[memory | pos hidden] operand")
            _same(g.args[1], wx, "[I | W2] weight")
            _check_gemm(g, "bf16", st, "gemm bf16 (Kp)")
            kp, mem = g.out.view(Bc, N, D), memory[:, :, :D]

        r1 = take("rows_linear")
        _same(r1.args[0], ln, "point_mlp input")
        _check_rows_linear(r1, st, "rows_linear mlp3")
        r2 = take("rows_linear")
        _same(r2.args[0], r1.out, "point_mlp layer 3 input")
        _check_rows_linear(r2, st, "rows_linear")
        tgt, current = r2.out, ln.clone()
        for i, (layer, head) in enumerate(zip(m.decoder_layers, m.reg_branches)):
            if big:
                q = take("query_pos_hidden")
                _same(q.args[2], current, f"layer {i} query pos input")
                _check_query_pos_hidden(q, st, "query_pos_hidden")
                qpos = lin(q.out, pe2.weight, pe2.bias, what=f"layer {i} pos_emb")
            else:
                r = take("rows_linear")
                _same(r.args[0], current, f"layer {i} query pos input")
                _check_rows_linear(r, st, "rows_linear mlp3")
                qpos = r.out
            sa = layer.self_attn
            qk = lin(tgt, sa.in_proj_weight[:2 * D], sa.in_proj_bias[:2 * D], add=qpos, what=f"layer {i} qk")
            v = lin(tgt, sa.in_proj_weight[2 * D:], sa.in_proj_bias[2 * D:], what=f"layer {i} v")
            a = take("self_attention32")
            _same(a.args[0], qk, f"layer {i} self attention qk")
            _same(a.args[1], v, f"layer {i} self attention v")
            ref, bound = _attn32_mirror(a.args[0][..., :D], a.args[0][..., D:], a.args[1], cross=False)
            st.check("self_attention32", _ratio(a.out, ref, bound))
            o = lin(a.out, sa.out_proj.weight, sa.out_proj.bias, what=f"layer {i} self out_proj")
            n = take("add_layernorm")
            _same(n.args[0], tgt, f"layer {i} norm1 x")
            _same(n.args[1], o, f"layer {i} norm1 y")
            _check_layernorm(n, st, "add_layernorm")
            tgt = n.out
            if tf32:
                ca = layer.cross_attn
                qh = lin(tgt, ca.in_proj_weight[:D], ca.in_proj_bias[:D], add=qpos, what=f"layer {i} cross q")
                c = take("cross_attention32")
                _same(c.args[0], qh, f"layer {i} cross attention q")
                _same(c.args[1], k_all[:, :, i * D:(i + 1) * D], f"layer {i} cross attention k")
                _same(c.args[2], v_all[:, :, i * D:(i + 1) * D], f"layer {i} cross attention v")
                ref, bound = _attn32_mirror(*c.args[:3], cross=True)
                st.check("cross_attention32", _ratio(c.out, ref, bound))
                att = lin(c.out, ca.out_proj.weight, ca.out_proj.bias, what=f"layer {i} cross out_proj")
            else:
                wqk, bqk, wvo, bvo, wvo16 = layers_w[i]
                qf = lin(tgt, wqk, bqk, out_dtype=torch.bfloat16, add=qpos, what=f"layer {i} folded queries")
                c = take("ctx_attention")
                _same(c.args[0], qf, f"layer {i} ctx_attention queries")
                _same(c.args[1], kp, f"layer {i} ctx_attention kp")
                _same(c.args[2], mem, f"layer {i} ctx_attention mem")
                _check_ctx(c, st, "ctx_attention")
                if big:
                    g = take("gemm_bias_act")
                    _same(g.args[0], c.out, f"layer {i} Wvo operand")
                    _same(g.args[1], wvo16, f"layer {i} Wvo bf16")
                    _same(g.args[2], bvo, f"layer {i} bvo")
                    _check_gemm(g, "bf16", st, "gemm bf16 (Wvo)")
                    att = g.out.view(Bc, 32, D)
                else:
                    r = take("rows_linear")
                    _same(r.args[0], c.out, f"layer {i} Wvo operand")
                    _same(r.args[1], wvo, f"layer {i} Wvo")
                    _check_rows_linear(r, st, "rows_linear")
                    att = r.out
            n = take("add_layernorm")
            _same(n.args[0], tgt, f"layer {i} norm2 x")
            _same(n.args[1], att, f"layer {i} norm2 y")
            _check_layernorm(n, st, "add_layernorm")
            tgt = n.out
            h1 = lin(tgt, layer.linear1.weight, layer.linear1.bias, relu=True, what=f"layer {i} linear1")
            ffn = lin(h1, layer.linear2.weight, layer.linear2.bias, what=f"layer {i} linear2")
            n = take("add_layernorm")
            _same(n.args[0], tgt, f"layer {i} norm3 x")
            _same(n.args[1], ffn, f"layer {i} norm3 y")
            _check_layernorm(n, st, "add_layernorm")
            tgt = n.out
            hid = lin(tgt, head[0].weight, head[0].bias, relu=True, what=f"layer {i} head")
            h = take("head_update")
            _same(h.args[0], hid, f"layer {i} head_update hidden")
            _same(h.args[3], current, f"layer {i} head_update current")
            _same(h.args[4], ln, f"layer {i} head_update noisy")
            _check_head_update(h, st, "head_update")
            _same(out[i, s0:s0 + chunk], h.out, f"layer {i}: the forward's output is the recorded cumulative offset")
            current = h.after
    assert next(it, None) is None, "calls left over"


# ------------------------------------------------------------------ tests: the recorded forward
FORWARD_CASES = [(1, 1024, "parity"), (7, 513, "parity"), (8, 300, "parity"), (16, 1024, "parity"), (8, 700, "realistic"),
                 (300, 129, "parity")]


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
@pytest.mark.parametrize("B,N,dist", FORWARD_CASES, ids=[f"b{b}_n{n}_{d}" for b, n, d in FORWARD_CASES])
def test_decoder_stages_match_fp64(dev, record, B, N, dist, prec):
    m = _model(prec, dev)
    ctx, line = (torch.from_numpy(a).to(dev) for a in synth.make_inputs(B, N, seed=B * 31 + N, dist=dist))
    with torch.no_grad():
        plain = m(ctx, line)           # also prepares every cached weight, so the recorded call issues only the forward
    out, calls = record(m, ctx, line)
    _same(out, plain, "the recorded forward is bit-identical to an unrecorded one")
    st = Stages(f"b{B}_n{N}_{dist}", prec)
    _walk(calls, m, prec, ctx, line, out, st)
    st.flush()


# ------------------------------------------------------------------ tests: prepared weights against the state dict
def _ulp_close(got, want64, what):
    got = got.detach().cpu().double().numpy()
    assert (np.abs(got - want64) <= np.spacing(np.abs(want64).astype(np.float32)).astype(np.float64)).all(), what


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
def test_prepared_weights_match_state_dict(dev, prec):
    sd = synth.make_state_dict(13)
    m = _model(prec, dev)
    with torch.no_grad():       # B = 8: 256 polyline rows, the tensor-core query side (TF32 weight copies in the tf32 tier)
        m(*(torch.from_numpy(a).to(dev) for a in synth.make_inputs(8, 300, seed=1)))
    f64 = lambda k: sd[k].astype(np.float64)
    scale = math.log2(math.e) / math.sqrt(32)
    layers, wx, b2 = m._attn_weights()
    for i, (wqk, bqk, wvo, bvo, wvo16) in enumerate(layers):
        p = f"decoder_layers.{i}.cross_attn."
        w, b = f64(p + "in_proj_weight"), f64(p + "in_proj_bias")
        wo, bo = f64(p + "out_proj.weight"), f64(p + "out_proj.bias")
        rq, rb, rv = np.zeros((8 * D, D)), np.zeros(8 * D), np.zeros((D, 8 * D))
        for h in range(8):
            Wq, Wk, Wv = (w[o + 32 * h:o + 32 * h + 32] for o in (0, D, 2 * D))
            rq[h * D:(h + 1) * D] = scale * Wk.T @ Wq
            rb[h * D:(h + 1) * D] = scale * b[32 * h:32 * h + 32] @ Wk
            rv[:, h * D:(h + 1) * D] = wo[:, 32 * h:32 * h + 32] @ Wv
        _ulp_close(wqk, rq, f"layer {i} Wqk")
        _ulp_close(bqk, rb, f"layer {i} bqk")
        _ulp_close(wvo, rv, f"layer {i} Wvo")
        _ulp_close(bvo, wo @ b[2 * D:] + bo, f"layer {i} bvo")
        _same(wvo16, wvo.bfloat16(), f"layer {i} Wvo (bf16) is Wvo rounded once")
    w2 = torch.from_numpy(sd["pos_emb.mlp.2.weight"]).to(dev)
    _same(wx, torch.cat([torch.eye(D, device=dev), w2.bfloat16().float()], 1).bfloat16(), "[I | W2]")
    _same(b2, torch.from_numpy(sd["pos_emb.mlp.2.bias"]).to(dev), "pos_emb layer 2 bias")

    for (w, b), (ci, bi) in zip(m._point_mlp_weights(), ((0, 1), (3, 4), (6, 7))):
        c, n = f"point_mlp.{ci}.", f"point_mlp.{bi}."
        s = f64(n + "weight") / np.sqrt(f64(n + "running_var") + m.point_mlp[bi].eps)
        _ulp_close(w, f64(c + "weight").reshape(s.shape[0], -1) * s[:, None], f"point_mlp.{ci} folded weight")
        _ulp_close(b, (f64(c + "bias") - f64(n + "running_mean")) * s + f64(n + "bias"), f"point_mlp.{ci} folded bias")

    wk, bk, wv, bv, w2r = m._kv_weights()
    t = lambda k: torch.from_numpy(sd[k]).to(dev)
    ipw = [t(f"decoder_layers.{i}.cross_attn.in_proj_weight") for i in range(6)]
    ipb = [t(f"decoder_layers.{i}.cross_attn.in_proj_bias") for i in range(6)]
    for got, want in ((wk, torch.cat([x[D:2 * D] for x in ipw])), (wv, torch.cat([x[2 * D:] for x in ipw])),
                      (w2r, t("pos_emb.mlp.2.weight"))):
        _tf32_exact(got, "K / V weight copy")
        _same(got, _rna_tf32(want), "K / V weight copies are the nearest TF32 values")
    _same(bk, torch.cat([x[D:2 * D] for x in ipb]), "K bias")
    _same(bv, torch.cat([x[2 * D:] for x in ipb]), "V bias")

    # the operand form of every tensor-core linear of the tf32 tier's query side
    used = [m.pos_emb.mlp[2].weight]
    for layer, head in zip(m.decoder_layers, m.reg_branches):
        sa, ca = layer.self_attn, layer.cross_attn
        used += [sa.in_proj_weight[:2 * D], sa.in_proj_weight[2 * D:], sa.out_proj.weight, ca.in_proj_weight[:D],
                 ca.out_proj.weight, layer.linear1.weight, layer.linear2.weight, head[0].weight]
    for w in used:
        got = m._tf32_weight(w)
        _tf32_exact(got, "TF32 weight copy")
        _same(got, _rna_tf32(w.detach()), "TF32 weight copies are the nearest TF32 values, not truncations")


# ------------------------------------------------------------------ tests: the attention kernels at their edges
def _legal_splits(N, upto=8):
    total = (N + 127) // 128
    return [s for s in range(1, min(total, upto) + 1) if (s - 1) * ((total + s - 1) // s) < total]


def _run_ctx(qf, kp, mem, splits):
    """lrn_ctx_attention into NaN-filled per-split outputs, then lrn_ctx_attention_merge into a NaN-filled result."""
    from pointnet_refine_b200 import ops
    B, N, _ = kp.shape
    dv = kp.device
    part = torch.full((B, splits, 256, 256), float("nan"), device=dv)
    lse = torch.full((B, splits, 256), float("nan"), device=dv)
    ops._call("lrn_ctx_attention", dv, qf, kp, 256, mem, 256, B, N, splits, part, 0, lse)
    merged = torch.full((B, 256, 256), float("nan"), device=dv)
    ops._call("lrn_ctx_attention_merge", dv, part, lse, B, splits, merged, 0)
    torch.cuda.synchronize()
    return part, lse, merged


def _check_ctx_kernel(qf, kp, mem, splits, case):
    from pointnet_refine_b200 import ops
    st = Stages(f"{case}_s{splits}", "bf16")
    part, lse, merged = _run_ctx(qf, kp, mem, splits)
    parts, ref, bound = _ctx_mirror(qf, kp, mem, splits)
    for s, (pref, pbound, lref, lbound) in enumerate(parts):
        st.check("ctx_attention split part", _ratio(part[:, s], pref, pbound + U * pref.abs()))
        st.check("ctx_attention split lse", _ratio(lse[:, s], lref, lbound))
    # the merge on its own inputs: w_s = 2^(lse_s - max) / sum, S FMAs
    L = lse.double()
    mx = L.amax(1, keepdim=True)
    w = torch.exp2(L - mx)
    w = w / w.sum(1, keepdim=True)
    werr = 2.0 ** -22 + LN2 * U * (L - mx).abs() + (splits + 2) * U
    wp = w[..., None] * part.double().abs()
    mref = (w[..., None] * part.double()).sum(1)
    mbound = (wp * (werr + werr.amax(1, keepdim=True))[..., None]).sum(1) + splits * U * wp.sum(1) + U * mref.abs()
    st.check("ctx_attention merge", _ratio(merged, mref, mbound))
    st.check("ctx_attention merged", _ratio(merged, ref, bound + U * ref.abs()))
    _same(ops.ctx_attention(qf, kp, mem, splits), part[:, 0] if splits == 1 else merged, f"{case}: ops.ctx_attention")
    st.flush()


def _gen(dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return lambda *s: torch.randn(*s, device=dev, generator=g)


@pytest.mark.parametrize("N", [129, 193, 255])
def test_ctx_attention_padding_isolation(dev, N):
    """Segment 0 scores near -60 (log2 units) on its own points, near 0 on segment 1's rows and on the zero fill past the
    last segment: a key admitted past the end of a segment would outweigh the real ones by 2^60."""
    r = _gen(dev, N)
    qf, kp, mem = 0.05 * r(2, 256, 256), r(2, N, 256), r(2, N, 256)
    qf[0, :, 0], kp[0, :, 0], kp[1, :, 0] = -7.5, 8.0, 0.0
    qf, kp, mem = qf.bfloat16(), kp.bfloat16(), mem.bfloat16()
    for splits in _legal_splits(N):
        _check_ctx_kernel(qf, kp, mem, splits, f"pad_b2_n{N}")


def test_ctx_attention_rescale_paths(dev):
    """Scores that rise by 8.25 per 128-point step (rescale every step), by 7.75 (every other step), by 127 (the old terms
    underflow to 0), and a decreasing ramp: four groups of 64 folded queries."""
    r = _gen(dev, 3)
    N = 1024
    qf, kp, mem = 0.002 * r(1, 256, 256), r(1, N, 256), r(1, N, 256)
    for gi, slope in enumerate((8.25, 7.75, 127.0, -8.25)):
        qf[0, 64 * gi:64 * gi + 64, 0] = slope
    kp[0, :, 0] = (torch.arange(N, device=dev) // 128).float()
    for splits in _legal_splits(N):
        _check_ctx_kernel(qf.bfloat16(), kp.bfloat16(), mem.bfloat16(), splits, "rescale_b1_n1024")


def test_ctx_attention_flat_and_dominant(dev):
    """qf = 0: every score equal, the output is the mean of mem and lse = log2(points).  Then one dominant point per
    segment at the step, half-step and split boundaries: the output is that point's row."""
    r = _gen(dev, 4)
    N = 1024
    mem = r(1, N, 256).bfloat16()
    kp = r(1, N, 256).bfloat16()
    qf = torch.zeros(1, 256, 256, device=dev).bfloat16()
    for splits in _legal_splits(N):
        _check_ctx_kernel(qf, kp, mem, splits, "flat_b1_n1024")
    pos = [0, 63, 64, 127, 128, 255, 256, 383, 384, 511, 512, 639, 640, 767, 768, 895, 896, N - 1]
    B = len(pos)
    qf, kp, mem = 0.01 * r(B, 256, 256), r(B, N, 256), r(B, N, 256)
    qf[:, :, 0], kp[:, :, 0] = 40.0, 0.0
    for b, p in enumerate(pos):
        kp[b, p, 0] = 1.0
    qf, kp, mem = qf.bfloat16(), kp.bfloat16(), mem.bfloat16()
    for splits in _legal_splits(N):
        _check_ctx_kernel(qf, kp, mem, splits, "dominant_b18_n1024")
        _, _, merged = _run_ctx(qf, kp, mem, splits)
        for b, p in enumerate(pos):
            assert float((merged[b] - mem[b, p].float()).abs().max()) <= 1e-3, (splits, p)


def test_ctx_attention_split_counts(dev):
    """Every legal split count at B = 1, N = 1024, and 40 splits of 65,536 points (more than one 32-lane group of
    splits in ctx_merge_kernel)."""
    r = _gen(dev, 5)
    for N, counts in ((1024, _legal_splits(1024)), (65536, [40])):
        qf = (r(1, 256, 256) / 16).bfloat16()
        mem = r(1, N, 256)
        kp = (mem + 0.5 * r(1, N, 256)).bfloat16()
        for splits in counts:
            _check_ctx_kernel(qf, kp, mem.bfloat16(), splits, f"splits_b1_n{N}")


@pytest.mark.parametrize("N,peaked", [(1, False), (31, False), (33, False), (255, False), (257, False), (1000, True)])
def test_cross_attention32_edges(dev, N, peaked):
    """Key counts that leave some of the eight warps without a key block, and a peaked ramp that forces the running
    rescale; k / v are column blocks of a wider buffer, as in the forward."""
    from pointnet_refine_b200 import ops
    r = _gen(dev, N)
    B = 3
    q = r(B, 32, 256) * (6.0 if peaked else 1.0)
    kall, vall = r(B, N, 6 * 256), r(B, N, 6 * 256)
    if peaked:
        kall = kall * torch.linspace(0.2, 3.0, N, device=dev)[None, :, None]
    st = Stages(f"cross32_b{B}_n{N}{'_peaked' if peaked else ''}", "tf32")
    for layer in (0, 5):
        k, v = kall[:, :, layer * 256:(layer + 1) * 256], vall[:, :, layer * 256:(layer + 1) * 256]
        got = ops.cross_attention32(q, k, v)
        ref, bound = _attn32_mirror(q, k, v, cross=True)
        st.check("cross_attention32", _ratio(got, ref, bound))
    st.flush()
