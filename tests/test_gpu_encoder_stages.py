"""The eval encoder checked stage by stage on its own intermediates, against fp64 references of the same arithmetic.

`test_gpu_parity.py` compares the encoder's outputs with the fp32 reference at 1e-2 of the output range (bf16 tier), which a
kernel that is subtly wrong (a truncating drain, a coarser gate factor, a bias one channel off, a dropped point in the
mean) still passes.  Here every stage is checked on the operands the kernels actually read:

  * the folded blob against the state dict (fold_linear_kernel),
  * the operand matrix `cat` of the last wave (conv1 + gate layer 1, conv2..conv5), read back from the caller-owned
    workspace, each column block against fp64 of the stored previous block,
  * `fused` against fp64 of the stored `cat` (fusion + gate), the point-major copy `fused_pm` against `fused`,
    `memory` (context_proj) against fp64 of `fused_pm`,
  * max / argmax / mean pooling against the kernel's own `fused`, on every pooling code path of the fusion epilogue.

Error bounds are derived from the arithmetic, not fitted.  With S = sum_k |a_k b_k| + |bias| in fp64 and `steps` the
number of MMA instructions along K, an fp32 accumulator that is truncated at every step is off by at most
acc = (steps + 2) * 2^-23 * S (the + 2: bias add and the epilogue's rounding of the sum).  A value then rounded into
an operand type is within acc + u * (|ref| + acc) of relu(ref), u being half an ulp relative to the value: 2^-8 for
bf16 (8 significant bits, round to nearest even), 2^-11 for TF32 (11 bits, round to nearest, ties away), 2^-22 for an
fp32x3 [hi | lo] pair (22 bits).  The worst error / bound ratio of every check is reported (parity_report.jsonl).
"""
import math

import numpy as np
import pytest
import torch

from oracle import lrn_oracle as orc
from oracle import synth
from tests.golden_util import report

pytestmark = pytest.mark.gpu

OUT_POOL, OUT_ARGMAX, OUT_FUSED, OUT_MEMORY = 1, 2, 4, 8          # LRN_OUT_* of include/lrn_b200.h
ALL_OUT = OUT_POOL | OUT_ARGMAX | OUT_FUSED | OUT_MEMORY
CHAN = (4, 64, 128, 256, 512, 1024)                               # kChan (csrc/lrn_abi.cu)
CAT_OFF = (0, 0, 64, 192, 448, 960)                               # kCatOff: column of feat_k in the operand row
DEFAULT_CHUNK_ROWS = 148 * 128 * 16                               # kDefaultChunkRows: 303,104 points per wave
WAVE_CUT_ROWS = 128 * 37 * 5                                      # 23,680: waves that end inside a segment
OPERAND = {"bf16": (2, 1), "tf32": (4, 1), "fp32x3": (4, 2)}      # element bytes, row width multiplier ([hi | lo])
TIERS = list(OPERAND)
MMA_K = {"bf16": 16, "tf32": 8, "fp32x3": 8}                      # K of one MMA instruction
PASSES = {"bf16": 1, "tf32": 1, "fp32x3": 3}                      # fp32x3: hi*hi + lo*hi + hi*lo
ROUND_U = {"bf16": 2.0 ** -8, "tf32": 2.0 ** -11, "fp32x3": 2.0 ** -22}   # half an ulp, relative
TINY = 2.0 ** -126                                                # below this, fp32 subnormal handling is not checked
# Gate factor gamma = 0.5 + 0.5 * sigmoid(z).  bf16 / tf32 tiers (gamma_pack, DESIGN.md section 3): held as the top 16
# mantissa bits of a float in [0.5, 1), rounded half up, so a step of 2^-17; the largest code is 1 - 2^-17, which is
# where every gamma above 1 - 2^-18 lands (the reference applies the same clamp).  Error: half a step plus the
# __expf / __fdividef approximation (2^-22).  fp32x3 tier: expf (2 ulp) and four correctly rounded operations.
GAMMA_TOP16 = 1.0 - 2.0 ** -17
GAMMA_ALLOW = {"bf16": 2.0 ** -18 + 2.0 ** -22, "tf32": 2.0 ** -18 + 2.0 ** -22, "fp32x3": 2.0 ** -21}
# Fraction of conv1 / gate layer 1 / conv2..conv5 outputs stored exactly as the fp64 result rounded to fp32 and then to
# the operand type (cases of >= 1000 points).  Measured on a B200: bf16 >= 0.9995 per layer, tf32 >= 0.996; fp32x3
# 0.48-0.50 for conv2..conv5 and 0.83 for conv1 (a 22-bit pair keeps most of the fp32 accumulator's last bits, so the
# accumulation order shows).
EXACT_FLOOR = {"bf16": 0.99, "tf32": 0.99, "fp32x3": 0.4}
ROW_BLOCK = 32768                                                # fp64 references in blocks of rows (bounded memory)


def _align(v, a):
    return (v + a - 1) // a * a


class PackedLayout:
    """Byte offsets of the folded blob; mirrors PackedLayout / packed_layout() in csrc/lrn_abi.cu.  Every entry starts
    on 1024 bytes; operand matrices are (Cout, Cin) K-major in the operand type, fp32x3 rows are [hi | lo]."""

    def __init__(self, prec):
        es, wm = OPERAND[prec]
        off = 0

        def take(nbytes):
            nonlocal off
            o, off = off, _align(off + nbytes, 1024)
            return o
        self.w1, self.b1, self.wg1, self.bg1 = take(64 * 4 * 4), take(64 * 4), take(64 * 4), take(64 * 4)   # fp32
        self.w = {k: take(CHAN[k] * CHAN[k - 1] * es * wm) for k in range(2, 6)}                             # conv2..5
        self.wfg = take(1024 * 2048 * es * wm)          # [fusion (1984 columns) | gate layer 2 (64 columns)]
        self.wp = take(256 * 1024 * es * wm)            # context_proj
        self.b = {k: take(CHAN[k] * 4) for k in range(2, 6)}
        self.bf, self.bg, self.bp = take(1024 * 4), take(1024 * 4), take(256 * 4)
        self.total = off


class WorkspaceLayout:
    """Byte offsets of the encoder workspace; mirrors WorkspaceLayout / workspace_layout() in csrc/lrn_abi.cu."""

    def __init__(self, B, N, prec, flags, chunk_rows):
        es, wm = OPERAND[prec]
        chunk = chunk_rows if chunk_rows > 0 else DEFAULT_CHUNK_ROWS
        self.chunk = min(_align(max(chunk, 128), 128), _align(B * N, 128))
        self.cat = 0                                                   # operand rows of the last wave: (chunk, 2048)
        off = _align(self.chunk * 2048 * es * wm, 1024)
        self.fused_pm = off                                            # point-major fused, LRN_OUT_MEMORY only
        if flags & OUT_MEMORY:
            off = _align(off + self.chunk * 1024 * es * wm, 1024)
        self.keys = off                                                # argmax keys, LRN_OUT_ARGMAX only
        if flags & OUT_ARGMAX:
            off = _align(off + B * 1024 * 8, 1024)
        self.total = off


# ------------------------------------------------------------------ operand types
def _dtype(prec):
    return torch.bfloat16 if prec == "bf16" else torch.float32


def _rna_tf32(x):
    """fp32 -> TF32, round to nearest with ties away from zero (cvt.rna.tf32.f32, low 13 bits cleared)."""
    return ((x.contiguous().view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)


def _to_operand(v, prec):
    """fp32 values as the tier stores them: bf16 (RNE), TF32 (RNA) or [hi | lo] TF32 pairs."""
    if prec == "bf16":
        return v.bfloat16()
    hi = _rna_tf32(v)
    return hi if prec == "tf32" else torch.cat([hi, _rna_tf32(v - hi)], -1)


def _cols(m, c0, c1, prec, width):
    """fp64 values of columns [c0, c1) of operand rows `m` ([hi | lo] halves of `width` columns for fp32x3)."""
    v = m[:, c0:c1].double()
    return v + m[:, width + c0:width + c1].double() if prec == "fp32x3" else v


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _check_split(m, width, what):
    """fp32x3 pairs: hi and lo are TF32-exact and lo is within half a TF32 ulp of hi (hi = rna(v), lo = rna(v - hi))."""
    hi, lo = m[:, :width], m[:, width:2 * width]
    assert ((_bits(hi) & 0x1FFF) == 0).all() and ((_bits(lo) & 0x1FFF) == 0).all(), what
    _, e = torch.frexp(hi)                                   # |hi| = f * 2^e, f in [0.5, 1): TF32 ulp 2^(e - 11)
    half_ulp = torch.ldexp(torch.ones_like(hi), e - 12)
    assert ((lo.abs() <= half_ulp) & ((hi != 0) | (lo == 0))).all(), what


def _round_back(v64, prec):
    """fp64 reference -> fp32 -> the tier's operand rounding, as fp64 (what a bit-exact kernel would store)."""
    r = _to_operand(v64.float(), prec)
    w = v64.shape[1]
    return r[:, :w].double() + r[:, w:].double() if prec == "fp32x3" else r.double()


def _check_linear(x, w, b, got, *, steps, u, relu=True, rounding=None, what=""):
    """got (R, C) fp64 = what the kernel stored for relu?(x @ w.T + b); x (R, K), w (C, K), b (C) fp64 operand values.
    Asserts |got - ref| <= acc + u (|ref| + acc); returns (worst error / bound, fraction stored bit-exact)."""
    worst, exact = 0.0, 0
    for r in range(0, x.shape[0], ROW_BLOCK):
        xs = x[r:r + ROW_BLOCK]
        ref = torch.addmm(b, xs, w.T)
        acc = (steps + 2) * 2.0 ** -23 * torch.addmm(b.abs(), xs.abs(), w.abs().T)
        want = ref.clamp_min(0) if relu else ref
        g = got[r:r + ROW_BLOCK]
        ratio = ((g - want).abs() / (acc + u * (ref.abs() + acc) + TINY)).nan_to_num(nan=math.inf)
        worst = max(worst, float(ratio.max()))
        exact += int((g == (rounding(want) if rounding else want.float().double())).sum())
    assert worst <= 1.0, f"{what}: error / bound = {worst:.3g}"
    return worst, exact / max(1, got.numel())


# ------------------------------------------------------------------ running the encoder on owned buffers
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _folded(sd, prec, dev):
    from pointnet_refine_b200 import ops
    enc = "context_encoder."
    t = {k[len(enc):]: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sd.items()
         if k.startswith(enc) and v.dtype == np.float32}
    t["context_proj.weight"] = torch.from_numpy(sd["context_proj.weight"]).to(dev)
    t["context_proj.bias"] = torch.from_numpy(sd["context_proj.bias"]).to(dev)
    return ops.FoldedEncoder(t, prec)


def _blob(folded, off, shape, dtype):
    n = math.prod(shape) * torch.empty(0, dtype=dtype).element_size()
    return folded.blob[off:off + n].view(dtype).view(shape)


def _forward(folded, ctx, flags, chunk_rows=0):
    """lrn_encoder_forward with a workspace this test owns (filled with NaN first: whatever a check reads was written
    by the kernels).  Returns the outputs, and for the last wave its first context row r0 and the workspace views
    `cat` (rows, 2048 * width multiplier) and `fused_pm` (rows, 1024 * width multiplier), row-major."""
    from pointnet_refine_b200 import ops
    from pointnet_refine_b200._lib import lib
    B, N, _ = ctx.shape
    prec, dev = folded.precision, ctx.device
    nbytes = lib.lrn_encoder_workspace_bytes(B, N, folded.prec_id, flags, chunk_rows)
    W = WorkspaceLayout(B, N, prec, flags, chunk_rows)
    assert nbytes == W.total
    ws = ops._aligned_bytes(nbytes, dev)
    ws.fill_(0xFF)
    nan = float("nan")
    out = {"global_feat": torch.full((B, 2048), nan, device=dev) if flags & (OUT_POOL | OUT_ARGMAX) else None,
           "argmax": torch.full((B, 1024), -1, dtype=torch.int64, device=dev) if flags & OUT_ARGMAX else None,
           "fused": torch.full((B, 1024, N), nan, device=dev) if flags & OUT_FUSED else None,
           "memory": torch.full((B, N, 256), nan, device=dev) if flags & OUT_MEMORY else None}
    ops._call("lrn_encoder_forward", dev, folded.blob, folded.prec_id, ctx, B, N, flags, out["global_feat"], out["fused"],
              out["argmax"], out["memory"], chunk_rows, ws, ws.numel())
    es, wm = OPERAND[prec]
    P = B * N
    r0 = (P - 1) // W.chunk * W.chunk                  # workspace rows [0, P - r0) hold context rows [r0, P)
    cat = ws[W.cat:W.cat + W.chunk * 2048 * es * wm].view(_dtype(prec))
    if prec == "bf16":   # tiled: [row tile of 128][column block of 64][128 rows][64 columns]
        cat = cat.view(W.chunk // 128, 32, 128, 64).permute(0, 2, 1, 3).reshape(W.chunk, 2048)
    else:
        cat = cat.view(W.chunk, 2048 * wm)
    out["r0"], out["cat"] = r0, cat[:P - r0]
    if flags & OUT_MEMORY:
        out["fused_pm"] = ws[W.fused_pm:W.fused_pm + W.chunk * 1024 * es * wm].view(_dtype(prec)).view(W.chunk, 1024 * wm)[:P - r0]
    torch.cuda.synchronize()
    return out


def _point_major(fused):
    B, C, N = fused.shape
    return fused.permute(0, 2, 1).reshape(B * N, C)


# ------------------------------------------------------------------ checks
def _record(case, prec, stage, ratio, exact=None):
    report(test="encoder_stages", case=case, tier=prec, stage=stage, ratio=ratio, exact=exact)


def _check_pooling(fused, gf, argmax, case, prec):
    """Pooled outputs against the kernel's own `fused`: max bit for bit (never -0.0), argmax the first maximal index,
    mean within the error of its fp32 summation: 31 sequential adds per warp (or a 5-level tree), the scaling by the
    rounded 1/N, then at most ceil(N/32) + 2 atomic adds of warp partials per (segment, channel); all terms >= 0."""
    B, _, N = fused.shape
    mx = fused.max(2).values
    assert torch.equal(_bits(gf[:, :1024]), _bits(mx)), case
    assert not (_bits(gf[:, :1024]) == -2 ** 31).any(), case
    if argmax is not None:
        idx = torch.arange(N, device=fused.device).expand_as(fused)
        first = torch.where(fused == mx[..., None], idx, N).min(2).values
        assert torch.equal(argmax, first), case
    mean64 = fused.double().mean(2)
    ratio = float(((gf[:, 1024:].double() - mean64).abs()
                   / ((math.ceil(N / 32) + 36) * 2.0 ** -24 * mean64 + TINY)).nan_to_num(nan=math.inf).max())
    _record(case, prec, "mean", ratio)
    assert ratio <= 1.0, (case, ratio)
    return mean64


def _check_stages(sd, ctx, prec, dev, case, chunk_rows=0):
    """Every stage of one encoder call (all outputs requested), each on the operands the kernels read."""
    folded = _folded(sd, prec, dev)
    L = PackedLayout(prec)
    B, N, _ = ctx.shape
    P = B * N
    out = _forward(folded, ctx, ALL_OUT, chunk_rows)
    r0, cat = out["r0"], out["cat"]
    _, wm = OPERAND[prec]
    dt = _dtype(prec)
    u = ROUND_U[prec]
    steps = lambda K: PASSES[prec] * K // MMA_K[prec]
    rnd = lambda v: _round_back(v, prec)
    f32 = lambda off, n: _blob(folded, off, (n,), torch.float32).double()
    res = {}

    # conv1 + gate layer 1: fp32 FMA chains (4 and 1 terms) on the raw points
    pts = ctx.reshape(P, 4)[r0:].double()
    w1 = _blob(folded, L.w1, (64, 4), torch.float32).double()
    x_int = pts[:, 3:4]
    wg1 = _blob(folded, L.wg1, (64, 1), torch.float32).double()
    if prec == "fp32x3":
        _check_split(cat, 2048, f"{case} operand rows")
    res["conv1"] = _check_linear(pts, w1, f32(L.b1, 64), _cols(cat, 0, 64, prec, 2048), steps=4, u=u, rounding=rnd,
                                 what=f"{case} {prec} conv1")
    res["gate1"] = _check_linear(x_int, wg1, f32(L.bg1, 64), _cols(cat, 1984, 2048, prec, 2048), steps=1, u=u,
                                 rounding=rnd, what=f"{case} {prec} gate layer 1")
    if prec == "bf16":   # the stand-alone first-layer kernel: same FMA chain, same rounding, bit for bit
        from pointnet_refine_b200 import ops
        pe = ops.point_embed(folded, ctx.reshape(P, 4)[r0:].contiguous(), tiled=True)
        for blk, c0 in ((0, 0), (31, 1984)):
            assert torch.equal(_bits(pe[:, blk].reshape(-1, 64)[:P - r0]), _bits(cat[:, c0:c0 + 64])), (case, blk)

    # conv2..conv5 on the stored previous column block
    for k in range(2, 6):
        w = _cols(_blob(folded, L.w[k], (CHAN[k], CHAN[k - 1] * wm), dt), 0, CHAN[k - 1], prec, CHAN[k - 1])
        x = _cols(cat, CAT_OFF[k - 1], CAT_OFF[k - 1] + CHAN[k - 1], prec, 2048)
        got = _cols(cat, CAT_OFF[k], CAT_OFF[k] + CHAN[k], prec, 2048)
        res[f"conv{k}"] = _check_linear(x, w, f32(L.b[k], CHAN[k]), got, steps=steps(CHAN[k - 1]), u=u, rounding=rnd,
                                        what=f"{case} {prec} conv{k}")

    # fusion + gate: fused = relu(X Wf^T + bf) * gamma(H Wg^T + bg) on the stored operand rows
    wfg = _blob(folded, L.wfg, (1024, 2048 * wm), dt)
    wf, wg = _cols(wfg, 0, 1984, prec, 2048), _cols(wfg, 1984, 2048, prec, 2048)
    bf, bg = f32(L.bf, 1024), f32(L.bg, 1024)
    fz = _point_major(out["fused"])
    worst, zmin, zmax = 0.0, math.inf, -math.inf
    for r in range(0, P - r0, ROW_BLOCK):
        x = _cols(cat[r:r + ROW_BLOCK], 0, 1984, prec, 2048)
        h = _cols(cat[r:r + ROW_BLOCK], 1984, 2048, prec, 2048)
        F = torch.addmm(bf, x, wf.T)
        acc_f = (steps(1984) + 2) * 2.0 ** -23 * torch.addmm(bf.abs(), x.abs(), wf.abs().T)
        z = torch.addmm(bg, h, wg.T)
        acc_z = (steps(64) + 2) * 2.0 ** -23 * torch.addmm(bg.abs(), h.abs(), wg.abs().T)
        zmin, zmax = min(zmin, float(z.min())), max(zmax, float(z.max()))
        gamma = 0.5 + 0.5 * torch.sigmoid(z)
        if prec != "fp32x3":
            gamma = gamma.clamp_max(GAMMA_TOP16)
        want = F.clamp_min(0) * gamma
        # d gamma / dz <= 1/8: the gate's own accumulation error moves gamma by at most acc_z / 8
        bound = acc_f * gamma + F.clamp_min(0) * (GAMMA_ALLOW[prec] + acc_z / 8) + 2.0 ** -24 * want + TINY
        ratio = ((fz[r0 + r:r0 + r + ROW_BLOCK].double() - want).abs() / bound).nan_to_num(nan=math.inf)
        worst = max(worst, float(ratio.max()))
    assert worst <= 1.0, f"{case} {prec} fusion: error / bound = {worst:.3g}"
    res["fusion"] = (worst, None)

    # point-major copy: the operand rounding of fused, bit for bit; context_proj on it (K = 1024, no ReLU)
    pm = out["fused_pm"]
    assert torch.equal(_bits(pm), _bits(_to_operand(fz[r0:].contiguous(), prec))), f"{case} {prec} fused_pm"
    x = _to_operand(fz, prec)
    x = x[:, :1024].double() + x[:, 1024:].double() if prec == "fp32x3" else x.double()
    wp = _cols(_blob(folded, L.wp, (256, 1024 * wm), dt), 0, 1024, prec, 1024)
    res["proj"] = _check_linear(x, wp, f32(L.bp, 256), out["memory"].reshape(P, 256).double(), steps=steps(1024), u=0.0,
                                relu=False, what=f"{case} {prec} context_proj")

    for stage, (ratio, exact) in res.items():
        _record(case, prec, stage, ratio, exact)
        if stage != "proj" and exact is not None and P - r0 >= 1000:
            assert exact >= EXACT_FLOOR[prec], (case, prec, stage, exact)
    out["mean64"] = _check_pooling(out["fused"], out["global_feat"], out["argmax"], case, prec)
    out["z_range"] = (zmin, zmax)
    return out


def _check_fold(sd, folded, prec):
    """The blob against the state dict, with fold_linear_kernel's fp32 operations (no fast-math: bit equality)."""
    L = PackedLayout(prec)
    _, wm = OPERAND[prec]
    enc = "context_encoder."
    eps = np.float32(1e-5)

    def stored(off, cout, cin, ld, col0=0):
        m = _blob(folded, off, (cout, ld * wm), _dtype(prec)).float()
        hi = m[:, col0:col0 + cin]
        return hi, (m[:, ld + col0:ld + col0 + cin] if prec == "fp32x3" else None)

    def expect(v):
        v = torch.from_numpy(np.ascontiguousarray(v)).to(folded.device)
        if prec == "bf16":
            return v.bfloat16().float(), None
        hi = _rna_tf32(v)
        return hi, (_rna_tf32(v - hi) if prec == "fp32x3" else None)

    def same(a, b, what):
        assert torch.equal(_bits(a[0]), _bits(b[0])), what
        if a[1] is not None:
            assert torch.equal(_bits(a[1]), _bits(b[1])), what + " (lo)"

    def folded_ref(conv, bn):
        w = sd[conv + ".weight"].reshape(sd[conv + ".weight"].shape[0], -1)
        s = sd[bn + ".weight"] / np.sqrt(sd[bn + ".running_var"] + eps)          # fp32, as sqrtf and IEEE division
        bias = (sd[conv + ".bias"] - sd[bn + ".running_mean"]).astype(np.float64) * s + sd[bn + ".bias"]
        return w * s[:, None], bias

    def bias_close(off, n, want, what):     # (b - mean) * s + beta contracts to one FMA: within 1 fp32 ulp
        got = _blob(folded, off, (n,), torch.float32).cpu().numpy().astype(np.float64)
        assert (np.abs(got - want) <= np.spacing(np.abs(want).astype(np.float32))).all(), what

    w1, b1 = folded_ref(enc + "conv1", enc + "bn1")                                # conv1 stays fp32, unrounded
    assert torch.equal(_bits(_blob(folded, L.w1, (64, 4), torch.float32).cpu()), torch.from_numpy(w1).view(torch.int32))
    bias_close(L.b1, 64, b1, "b1")
    for name, off in (("weight", L.wg1), ("bias", L.bg1)):                        # gate layer 1: copied
        got = _blob(folded, off, (64,), torch.float32).cpu()
        assert torch.equal(_bits(got), torch.from_numpy(sd[enc + "intensity_gate.0." + name].reshape(64)).view(torch.int32))
    for k in range(2, 6):
        w, b = folded_ref(f"{enc}conv{k}", f"{enc}bn{k}")
        same(stored(L.w[k], CHAN[k], CHAN[k - 1], CHAN[k - 1]), expect(w), f"{prec} conv{k} weights")
        bias_close(L.b[k], CHAN[k], b, f"{prec} conv{k} bias")
    w, b = folded_ref(enc + "fusion.0", enc + "fusion.1")
    same(stored(L.wfg, 1024, 1984, 2048), expect(w), f"{prec} fusion weights")
    bias_close(L.bf, 1024, b, f"{prec} fusion bias")
    same(stored(L.wfg, 1024, 64, 2048, 1984), expect(sd[enc + "intensity_gate.2.weight"].reshape(1024, 64)),
         f"{prec} gate layer 2 weights (columns 1984..2047)")
    same(stored(L.wp, 256, 1024, 1024), expect(sd["context_proj.weight"]), f"{prec} context_proj weights")
    for off, n, key in ((L.bg, 1024, enc + "intensity_gate.2.bias"), (L.bp, 256, "context_proj.bias")):
        assert torch.equal(_bits(_blob(folded, off, (n,), torch.float32).cpu()), torch.from_numpy(sd[key]).view(torch.int32))


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("prec", TIERS)
def test_fold_matches_state_dict(dev, prec):
    for sd in (synth.make_state_dict(11), _edge_state_dict()[0]):
        _check_fold(sd, _folded(sd, prec, dev), prec)


@pytest.mark.parametrize("prec", TIERS)
@pytest.mark.parametrize("B,N", [(1, 1), (1, 127), (1, 129), (3, 1000), (2, 4096)])
def test_stages_match_fp64(dev, B, N, prec):
    sd = synth.make_state_dict(11)
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=77)[0]).to(dev)
    _check_stages(sd, ctx, prec, dev, f"b{B}_n{N}")


@pytest.mark.parametrize("prec", TIERS)
def test_stages_realistic_inputs(dev, prec):
    """Metres and integer intensity counts (0..255): the first layer sees large, exactly representable inputs."""
    sd = synth.make_state_dict(3)
    ctx = torch.from_numpy(synth.make_inputs(3, 1000, seed=5, dist="realistic")[0]).to(dev)
    _check_stages(sd, ctx, prec, dev, "b3_n1000_realistic")


def _edge_state_dict():
    """State dict and inputs for the input edges: segment 1 repeats one point, segment 2 is all zeros; at the zero point
    conv1 channels 0..7 and fused channels 0..63 are ReLU-dead (pre-activation -0.05, live elsewhere); gate layer 2 is
    scaled so that its pre-activation reaches +-40 (gamma at both ends of its range)."""
    enc = "context_encoder."
    sd = synth.make_state_dict(7)
    ctx = synth.make_inputs(4, 300, seed=9)[0]
    ctx[1] = ctx[1, :1]
    ctx[2] = 0.0
    w1, b1 = orc.fold_bn(sd, enc + "conv1", enc + "bn1", np.float64)
    sd[enc + "bn1.bias"][:8] -= (b1[:8] + 0.05).astype(np.float32)
    _, _, _, feats = orc.encoder_forward(sd, np.zeros((1, 1, 4), np.float32), np.float64, return_feats=True)
    wf, bf = orc.fold_bn(sd, enc + "fusion.0", enc + "fusion.1", np.float64)
    f0 = np.concatenate([f.reshape(1, -1) for f in feats], 1) @ wf.T + bf
    sd[enc + "fusion.1.bias"][:64] -= (f0[0, :64] + 0.05).astype(np.float32)
    h = np.maximum(ctx[..., 3:4].reshape(-1, 1).astype(np.float64) @ sd[enc + "intensity_gate.0.weight"].reshape(64, 1).T
                   + sd[enc + "intensity_gate.0.bias"], 0)
    z = h @ sd[enc + "intensity_gate.2.weight"].reshape(1024, 64).T.astype(np.float64) + sd[enc + "intensity_gate.2.bias"]
    k = np.float32(40.0 / np.abs(z).max())
    sd[enc + "intensity_gate.2.weight"] *= k
    sd[enc + "intensity_gate.2.bias"] *= k
    return sd, ctx


@pytest.mark.parametrize("prec", TIERS)
def test_stages_input_edges(dev, prec):
    sd, ctx = _edge_state_dict()
    out = _check_stages(sd, torch.from_numpy(ctx).to(dev), prec, dev, "b4_n300_edges")
    zmin, zmax = out["z_range"]
    assert zmin < -12 and zmax > 12, out["z_range"]      # both ends: gamma = 0.5 and gamma above 1 - 2^-18
    fused, gf, am = out["fused"], out["global_feat"], out["argmax"]
    assert torch.equal(fused[1], fused[1, :, :1].expand_as(fused[1]))        # identical points, identical features
    assert (am[1] == 0).all() and (am[2] == 0).all()                         # every channel ties: the first point
    assert (_bits(gf[2, :64]) == 0).all() and (_bits(gf[2, 1024:1088]) == 0).all()   # dead: +0.0 max and mean
    assert (gf[0, :64] > 0).any()                                            # ... while live on ordinary points


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
def test_stages_full_default_wave(dev, prec):
    """74 x 4096 = 303,104 points: one full default wave, 16 tiles per CTA pair.  Only at this size does the chain kernel's
    rotating weight-stage ring pass through every position; every row of every stage is checked."""
    sd = synth.make_state_dict(2)
    ctx = torch.randn(74, 4096, 4, device=dev, generator=torch.Generator(device=dev).manual_seed(13))
    out = _check_stages(sd, ctx, prec, dev, "b74_n4096_wave")
    assert out["r0"] == 0 and out["cat"].shape[0] == 74 * 4096


# Pooling: the fusion epilogue has four paths.  "fast" (no argmax, N % 32 == 0: every warp's 32 points in one
# segment); GENERAL with a uniform warp pooled through shared memory ("smem") or with argmax keys ("argmax"); and the
# per-segment loop of a warp that straddles segments or the end of the points ("straddle").
POOL_CASES = [
    (7, 1, 0, "straddle"), (5, 3, 0, "straddle"), (9, 31, 0, "straddle"), (6, 32, 0, "fast+argmax"),
    (5, 33, 0, "smem+argmax+straddle"), (3, 37, 0, "smem+argmax+straddle"), (3, 300, 0, "smem+argmax+straddle"),
    (2, 4096, 0, "fast+argmax"), (9, 4096, WAVE_CUT_ROWS, "fast+argmax-wavecut"),
    (11, 3000, WAVE_CUT_ROWS, "smem+argmax+straddle-wavecut"),
]


@pytest.mark.parametrize("prec", TIERS)
@pytest.mark.parametrize("B,N,chunk_rows,paths", POOL_CASES, ids=[f"b{b}_n{n}_{p}" for b, n, _, p in POOL_CASES])
def test_pooling_matches_own_fused(dev, B, N, chunk_rows, paths, prec):
    """Max / argmax / mean against the kernel's own fused output; then the same call without fused (the product's
    configuration), with and without argmax: max bit-identical, mean within the same bound."""
    sd = synth.make_state_dict(11)
    folded = _folded(sd, prec, dev)
    ctx = torch.from_numpy(synth.make_inputs(B, N, seed=B * 7919 + N)[0]).to(dev)
    full = _forward(folded, ctx, OUT_POOL | OUT_ARGMAX | OUT_FUSED, chunk_rows)
    case = f"pool_b{B}_n{N}_{paths}"
    mean64 = _check_pooling(full["fused"], full["global_feat"], full["argmax"], case, prec)
    bound = (math.ceil(N / 32) + 36) * 2.0 ** -24 * mean64 + TINY
    for flags in (OUT_POOL, OUT_POOL | OUT_ARGMAX):
        o = _forward(folded, ctx, flags, chunk_rows)
        gf = o["global_feat"]
        assert torch.equal(_bits(gf[:, :1024]), _bits(full["global_feat"][:, :1024])), (case, flags)
        ratio = float(((gf[:, 1024:].double() - mean64).abs() / bound).max())
        _record(case, prec, f"mean_flags{flags}", ratio)
        assert ratio <= 1.0, (case, flags, ratio)
        if flags & OUT_ARGMAX:
            assert torch.equal(o["argmax"], full["argmax"]), case


@pytest.mark.parametrize("prec", TIERS)
def test_fused_is_wave_invariant(dev, prec):
    """Every output element is computed by one tile in the same k order whatever the wave size: fused is bit-identical
    between the default waves and waves that end inside segments (9 x 4096 points: two waves of 23,680 rows)."""
    sd = synth.make_state_dict(4)
    folded = _folded(sd, prec, dev)
    ctx = torch.from_numpy(synth.make_inputs(9, 4096, seed=3)[0]).to(dev)
    a = _forward(folded, ctx, OUT_FUSED)["fused"]
    b = _forward(folded, ctx, OUT_FUSED, WAVE_CUT_ROWS)["fused"]
    assert torch.equal(_bits(a), _bits(b))
