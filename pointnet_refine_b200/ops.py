"""Host-side operator wrappers: torch tensors in, C-ABI calls (raw device pointers + the current
CUDA stream) out.  PyTorch is only the allocator / stream provider here."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import OUT_ARGMAX, OUT_FUSED, OUT_MEMORY, OUT_MEMORY_BF16, OUT_POOL, PRECISIONS, lib

DEFAULT_CHUNK_ROWS = 148 * 128 * 16   # keep in sync with kDefaultChunkRows (csrc/lrn_abi.cu)


def _call(fn: str, device, *args) -> None:
    """lib.<fn>(*args, stream) on `device` and its current stream: a tensor is passed as its data pointer, None as NULL;
    a non-zero status raises RuntimeError."""
    with torch.cuda.device(device):
        args = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]
        _lib.check(getattr(lib, fn)(*args, torch.cuda.current_stream(device).cuda_stream), fn)


def _aligned_bytes(nbytes: int, device, align: int = 1024):
    """uint8 buffer whose data pointer is `align`-byte aligned."""
    raw = torch.empty(nbytes + align, dtype=torch.uint8, device=device)
    off = (-raw.data_ptr()) % align
    return raw[off:off + nbytes]


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32 or not t.is_cuda:
        raise TypeError("expected a float32 CUDA tensor")
    return t.contiguous()


class FoldedEncoder:
    """Device blob with the BN-folded, K-major operand matrices of one precision tier
    (lrn_encoder_fold).  Keeps references to nothing: it is a snapshot of the parameters."""

    def __init__(self, tensors: dict, precision: str, bn_eps: float = 1e-5):
        """tensors: the reference state_dict entries of `context_encoder.*` (prefix stripped) and,
        optionally, `context_proj.weight` / `context_proj.bias`; float32 CUDA tensors."""
        self.precision = precision
        self.prec_id = PRECISIONS[precision]
        dev = tensors["conv1.weight"].device
        self.device = dev
        keep = []

        def ptr(name):
            t = _f32c(tensors[name].detach())
            keep.append(t)
            return t.data_ptr()

        p = _lib.EncoderParams()
        for k in range(5):
            p.conv_w[k] = ptr(f"conv{k + 1}.weight")
            p.conv_b[k] = ptr(f"conv{k + 1}.bias")
            p.bn_w[k] = ptr(f"bn{k + 1}.weight")
            p.bn_b[k] = ptr(f"bn{k + 1}.bias")
            p.bn_mean[k] = ptr(f"bn{k + 1}.running_mean")
            p.bn_var[k] = ptr(f"bn{k + 1}.running_var")
        p.fusion_w, p.fusion_b = ptr("fusion.0.weight"), ptr("fusion.0.bias")
        p.fusion_bn_w, p.fusion_bn_b = ptr("fusion.1.weight"), ptr("fusion.1.bias")
        p.fusion_bn_mean, p.fusion_bn_var = ptr("fusion.1.running_mean"), ptr("fusion.1.running_var")
        p.gate0_w, p.gate0_b = ptr("intensity_gate.0.weight"), ptr("intensity_gate.0.bias")
        p.gate2_w, p.gate2_b = ptr("intensity_gate.2.weight"), ptr("intensity_gate.2.bias")
        self.has_proj = "context_proj.weight" in tensors
        if self.has_proj:
            p.proj_w, p.proj_b = ptr("context_proj.weight"), ptr("context_proj.bias")
        p.bn_eps = bn_eps
        nbytes = lib.lrn_encoder_packed_bytes(self.prec_id)
        self.blob = _aligned_bytes(nbytes, dev)
        _call("lrn_encoder_fold", dev, C.byref(p), self.prec_id, self.blob, nbytes)
        del keep


_workspaces: dict = {}


def _workspace(nbytes: int, device):
    """Grow-only scratch buffer per (device, stream): calls on different streams never share one, and a buffer that has
    been replaced by a larger one stays alive for whoever still holds it (graph.py keeps the one its capture baked in)."""
    key = (device.type, device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        _workspaces[key] = ws = _aligned_bytes(nbytes, device)
    return ws


def workspaces_of(device) -> list:
    """The scratch buffers currently cached for `device` (a CUDA graph must keep the ones it captured alive)."""
    return [ws for key, ws in _workspaces.items() if key[:2] == (device.type, device.index)]


def encoder_forward(folded: FoldedEncoder, context: torch.Tensor, *, pool=True, argmax=False, fused=False,
                    memory=False, memory_bf16=False, chunk_rows: int = 0):
    """Run the fused encoder on context (B, N, 4) float32 CUDA.  Returns a dict with the requested
    outputs: global_feat (B,2048), argmax (B,1024) int64, fused (B,1024,N), memory (B,N,256).
    memory_bf16 (bf16 tier): memory is returned as a (B,N,512) bfloat16 buffer whose columns [0,256) hold it and
    whose columns [256,512) are uninitialised (filled by pos_hidden for the decoder's context side)."""
    if context.dim() != 3 or context.shape[-1] != 4:
        raise ValueError(f"context must be (B, N, 4), got {tuple(context.shape)}")
    context = _f32c(context)
    B, N, _ = context.shape
    if B == 0 or N == 0:
        raise ValueError("empty context (the reference's torch.max over an empty dimension raises too)")
    dev = context.device
    flags = (OUT_POOL if pool else 0) | (OUT_ARGMAX if argmax else 0) | (OUT_FUSED if fused else 0) | \
            (OUT_MEMORY if memory else 0) | (OUT_MEMORY_BF16 if memory and memory_bf16 else 0)
    if memory and not folded.has_proj:
        raise ValueError("memory output needs context_proj weights in the folded blob")
    out = {}
    gf = fz = am = mem = None
    if pool or argmax:
        out["global_feat"] = gf = torch.empty(B, 2048, dtype=torch.float32, device=dev)
    if argmax:
        out["argmax"] = am = torch.empty(B, 1024, dtype=torch.int64, device=dev)
    if fused:
        out["fused"] = fz = torch.empty(B, 1024, N, dtype=torch.float32, device=dev)
    if memory:
        out["memory"] = mem = (torch.empty(B, N, 512, dtype=torch.bfloat16, device=dev) if memory_bf16 else
                               torch.empty(B, N, 256, dtype=torch.float32, device=dev))
    nbytes = lib.lrn_encoder_workspace_bytes(B, N, folded.prec_id, flags, chunk_rows)
    ws = _workspace(nbytes, dev)
    _call("lrn_encoder_forward", dev, folded.blob, folded.prec_id, context, B, N, flags, gf, fz, am, mem, chunk_rows, ws,
          ws.numel())
    return out


def _cum_out(out, current):
    if out is None:
        return torch.empty_like(current)
    if out.shape != current.shape or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError("out must be a contiguous float32 tensor of current's shape")
    return out


def head_forward(w1, b1, w2, b2, tgt, current, noisy, out=None):
    """reg_branches[i] + cumulative-offset update (lrn_head_forward).  `current` (B,M,3) is updated
    in place; returns the cumulative offset (B,M,3) (written into `out` when given)."""
    tgt = _f32c(tgt)
    rows = tgt.numel() // 256
    cum = _cum_out(out, current)
    _call("lrn_head_forward", tgt.device, _f32c(w1), _f32c(b1), _f32c(w2), _f32c(b2), tgt, rows, current, _f32c(noisy), cum)
    return cum


def gemm_bias_act(a: torch.Tensor, w: torch.Tensor, bias, *, relu=False, out_dtype=None):
    """out = act(a @ w.T + bias) on the tcgen05 path.  a (M,K), w (N,K): both bfloat16 (bf16 tier) or
    both float32 (tf32 tier)."""
    if a.dtype != w.dtype or a.dtype not in (torch.bfloat16, torch.float32):
        raise TypeError("a and w must both be bfloat16 or float32")
    prec = _lib.PREC_BF16 if a.dtype == torch.bfloat16 else _lib.PREC_TF32
    a, w = a.contiguous(), w.contiguous()
    M, K = a.shape
    N = w.shape[0]
    out_dtype = out_dtype or (torch.float32 if prec == _lib.PREC_TF32 else torch.bfloat16)
    out = torch.empty(M, N, dtype=out_dtype, device=a.device)
    b = bias.contiguous().float() if bias is not None else None
    _call("lrn_gemm_bias_act", a.device, prec, a, K, w, K, b, out, N, int(out_dtype == torch.float32), int(relu), M, N, K)
    return out


def profile_enable(on: bool) -> None:
    _lib.check(lib.lrn_profile_enable(int(on)), "lrn_profile_enable")


def profile_read() -> dict:
    """{stage: (milliseconds, launches)} accumulated since the previous read (syncs on the events)."""
    ms = (C.c_float * len(_lib.STAGES))()
    n = (C.c_int64 * len(_lib.STAGES))()
    _lib.check(lib.lrn_profile_read(ms, n), "lrn_profile_read")
    return {name: (float(ms[i]), int(n[i])) for i, name in enumerate(_lib.STAGES)}


def gemm_tn(at: torch.Tensor, bt: torch.Tensor) -> torch.Tensor:
    """out (M,N) fp32 = at.T @ bt for bf16 at (K,M), bt (K,N) row-major (MN-major tcgen05 operands, split-K)."""
    if at.dtype != torch.bfloat16 or bt.dtype != torch.bfloat16:
        raise TypeError("bfloat16 operands expected")
    K, M = at.shape
    N = bt.shape[1]
    out = torch.empty(M, N, dtype=torch.float32, device=at.device)
    _call("lrn_gemm_tn", at.device, at, at.stride(0), bt, bt.stride(0), out, N, M, N, K)
    return out


def ctx_attention(qfold: torch.Tensor, kp: torch.Tensor, mem: torch.Tensor, splits: int | None = None,
                  out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """softmax(qfold @ kp^T) @ mem per segment on the tensor cores, K / V never materialised (lrn_ctx_attention).
    qfold (B, 256, 256) bf16 folded queries (scores in log2 units), kp / mem (B, N, 256) bf16 (rows may be strided
    views of a wider buffer) -> (B, 256, 256) in out_dtype (fp32, or bf16 written straight from the kernel when a
    segment is not split)."""
    for t in (qfold, kp, mem):
        if t.dtype != torch.bfloat16 or not t.is_cuda:
            raise TypeError("ctx_attention expects CUDA bfloat16 tensors")
    B, N, d = kp.shape
    if d != 256 or tuple(qfold.shape) != (B, 256, 256) or mem.shape != kp.shape:
        raise ValueError(f"ctx_attention shapes: qfold {tuple(qfold.shape)}, kp {tuple(kp.shape)}, mem {tuple(mem.shape)}")

    def rows(t):  # (B, N, 256) view with unit column stride and segments back to back -> row pitch
        if t.stride(2) != 1 or (B > 1 and t.stride(0) != N * t.stride(1)):
            t = t.contiguous()
        return t, t.stride(1)
    qfold = qfold.contiguous()
    (kp, ld_kp), (mem, ld_mem) = rows(kp), rows(mem)
    if splits is None:
        splits = lib.lrn_ctx_attention_splits(B, N)
    direct_bf16 = out_dtype == torch.bfloat16 and splits == 1
    out = torch.empty(B, splits, 256, 256, dtype=torch.bfloat16 if direct_bf16 else torch.float32, device=kp.device)
    lse = torch.empty(B, splits, 256, dtype=torch.float32, device=kp.device)
    _call("lrn_ctx_attention", kp.device, qfold, kp, ld_kp, mem, ld_mem, B, N, splits, out, int(direct_bf16), lse)
    if splits == 1 and (direct_bf16 or out_dtype == torch.float32):
        return out[:, 0]
    merged = torch.empty(B, 256, 256, dtype=out_dtype, device=kp.device)     # merge the splits by their log-sum-exp
    _call("lrn_ctx_attention_merge", kp.device, out, lse, B, splits, merged, int(out_dtype == torch.bfloat16))
    return merged


def pos_hidden(w1: torch.Tensor, b1: torch.Tensor, context: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[..., :] = bf16(relu(context[..., :3] @ w1.T + b1)) (lrn_pos_hidden); `out` is a (B, N, 256) bf16 view whose
    rows may be strided (e.g. columns [256,512) of encoder_forward's memory_bf16 buffer)."""
    context = _f32c(context)
    P = context.numel() // 4
    if out.dtype != torch.bfloat16 or out.shape[-1] != 256 or out.stride(-1) != 1 or out.numel() != P * 256:
        raise ValueError("pos_hidden: out must be a bfloat16 (..., 256) view with unit column stride")
    ld = out.stride(-2)
    if out.dim() == 3 and out.shape[0] > 1 and out.stride(0) != out.shape[1] * ld:
        raise ValueError("pos_hidden: segments of `out` must be back to back")
    _call("lrn_pos_hidden", context.device, _f32c(w1), _f32c(b1), context, P, out, ld)
    return out


def add_layernorm(x: torch.Tensor, y, norm: torch.nn.LayerNorm) -> torch.Tensor:
    """norm(x + y) for fp32 (..., 256) tensors in one kernel (lrn_add_layernorm); y may be None."""
    x = _f32c(x)
    y = _f32c(y) if y is not None else None
    out = torch.empty_like(x)
    _call("lrn_add_layernorm", x.device, x, y, _f32c(norm.weight.detach()), _f32c(norm.bias.detach()), float(norm.eps), out, None,
          x.numel() // x.shape[-1], x.shape[-1])
    return out


def self_attention32(qk: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """Softmax attention among the 32 polyline points of every segment, 8 heads x 32 (lrn_self_attention32):
    qk (B, 32, 512) = [q | k] projections, v (B, 32, 256) -> (B, 32, 256), heads concatenated."""
    qk, v = _f32c(qk), _f32c(v)
    B = qk.shape[0]
    if tuple(qk.shape) != (B, 32, 512) or tuple(v.shape) != (B, 32, 256):
        raise ValueError(f"self_attention32 shapes {tuple(qk.shape)}, {tuple(v.shape)}")
    out = torch.empty_like(v)
    _call("lrn_self_attention32", v.device, qk, v, out, B)
    return out


def head_update(hidden: torch.Tensor, w2, b2, current: torch.Tensor, noisy: torch.Tensor, out=None) -> torch.Tensor:
    """Second head layer + cumulative-offset update (lrn_head_update): `current` (B,M,3) is updated in place; returns the
    cumulative offset (B,M,3) (written into `out` when given)."""
    hidden = _f32c(hidden)
    rows = hidden.numel() // 128
    cum = _cum_out(out, current)
    _call("lrn_head_update", hidden.device, hidden, _f32c(w2.detach()), _f32c(b2.detach()), rows, current, _f32c(noisy), cum)
    return cum


def rows_linear(x: torch.Tensor, w: torch.Tensor, bias, *, add: torch.Tensor | None = None, mlp3=None, relu=False,
                out_dtype=torch.float32) -> torch.Tensor:
    """nn.Linear for FEW rows in fp32 FMA (lrn_rows_linear): out (M, N) = act(x' @ w.T + bias), w (N, K) fp32.
    x' = x (M, K), or x + add, or relu(c @ w1.T + b1) with x = c (M, 3) and mlp3 = (w1 (K,3), b1 (K)): the K = 3 first
    layer of pos_emb / point_mlp fused into the operand load.  Leading dimensions of x are flattened."""
    w = _f32c(w.detach())
    N, K = w.shape
    w1 = b1 = None
    lead = x.shape[:-1]
    x = _f32c(x).reshape(-1, x.shape[-1])
    M = x.shape[0]
    if mlp3 is not None:
        if x.shape[1] != 3 or add is not None:
            raise ValueError("rows_linear: mlp3 takes (M, 3) coordinates and no addend")
        w1, b1 = _f32c(mlp3[0].detach()).reshape(-1, 3), _f32c(mlp3[1].detach())
        if w1.shape[0] != K or b1.numel() != K:
            raise ValueError("rows_linear: mlp3 first layer must have K outputs")
    elif x.shape[1] != K:
        raise ValueError(f"rows_linear: x has {x.shape[1]} columns, w expects {K}")
    x2 = None
    if add is not None:
        x2 = _f32c(add).reshape(-1, K)
        if x2.shape[0] != M:
            raise ValueError("rows_linear: addend shape")
    b = _f32c(bias.detach()) if bias is not None else None
    out = torch.empty(M, N, dtype=out_dtype, device=x.device)
    _call("lrn_rows_linear", x.device, x, x.stride(0), x2, K, w1, b1, w, b, out, N, int(out_dtype == torch.bfloat16), int(relu),
          M, N, K)
    return out.view(*lead, N)


def query_pos_hidden(w1: torch.Tensor, b1: torch.Tensor, coords: torch.Tensor, round_tf32: bool = False) -> torch.Tensor:
    """relu(coords[..., :3] @ w1.T + b1): (..., 3 or 4) -> (..., 256) fp32 (lrn_query_pos_hidden), first layer of pos_emb on the
    polyline points (rows of 3) or the context points (rows of 4); optionally rounded to the nearest TF32 value."""
    coords = _f32c(coords)
    ld = coords.shape[-1]
    rows = coords.numel() // ld
    out = torch.empty(*coords.shape[:-1], 256, dtype=torch.float32, device=coords.device)
    _call("lrn_query_pos_hidden", coords.device, _f32c(w1.detach()), _f32c(b1.detach()), coords, ld, rows, out, int(round_tf32))
    return out


def add(a: torch.Tensor, b: torch.Tensor | None, round_tf32: bool = False) -> torch.Tensor:
    """a + b for fp32 tensors of equal shape (lrn_add); b = None copies; round_tf32 rounds to the nearest TF32 value."""
    a = _f32c(a)
    b = _f32c(b) if b is not None else None
    if (b is not None and a.shape != b.shape) or a.numel() % 4:
        raise ValueError("add: equal shapes with a multiple of 4 elements expected")
    out = torch.empty_like(a)
    _call("lrn_add", a.device, a, b, out, a.numel(), int(round_tf32))
    return out


def cross_attention32(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """fp32 cross attention of 32 queries per segment over N points, 8 heads x 32 (lrn_cross_attention32):
    q (B, 32, 256); k, v (B, N, 256) views with unit column stride whose rows may be strided (a layer's column block of
    the hoisted (B, N, L*256) projections) -> (B, 32, 256)."""
    q = _f32c(q)
    B, N, d = k.shape
    if tuple(q.shape) != (B, 32, 256) or d != 256 or v.shape != k.shape:
        raise ValueError(f"cross_attention32 shapes {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    for t in (k, v):
        if t.dtype != torch.float32 or t.stride(2) != 1 or (B > 1 and t.stride(0) != N * t.stride(1)):
            raise ValueError("cross_attention32: k / v must be fp32 (B, N, 256) views with segments back to back")
    if k.stride(1) != v.stride(1):
        raise ValueError("cross_attention32: k and v must share their row pitch")
    out = torch.empty(B, 32, 256, dtype=torch.float32, device=q.device)
    _call("lrn_cross_attention32", q.device, q, k, v, k.stride(1), B, N, out)
    return out


def point_embed(folded: FoldedEncoder, context: torch.Tensor, tiled: bool = False, out: torch.Tensor | None = None) -> torch.Tensor:
    """Stand-alone first layer (+ gate layer 1): context (P, 4) or (B, N, 4) fp32 -> operand rows (P, 2048) in the
    tier's operand type with columns [0,64) and [1984,2048) written (the rest is left uninitialised).
    tiled (bf16 tier): the result is the tiled operand matrix of the default path instead,
    (ceil(P/128), 32, 128, 64): [row tile][column block][row][column]; blocks 0 and 31 are written.
    `out`: a buffer returned by an earlier call with the same arguments, to be reused."""
    context = _f32c(context).reshape(-1, 4)
    P = context.shape[0]
    dt = torch.float32 if folded.precision == "tf32" else torch.bfloat16
    shape = ((P + 127) // 128, 32, 128, 64) if tiled else (P, 2048)
    if out is None:
        out = torch.empty(shape, dtype=dt, device=context.device)
    elif tuple(out.shape) != shape or out.dtype != dt or not out.is_contiguous():
        raise ValueError("point_embed: `out` does not match the requested layout")
    _call("lrn_point_embed", context.device, folded.blob, folded.prec_id, context, P, out, int(tiled))
    return out
