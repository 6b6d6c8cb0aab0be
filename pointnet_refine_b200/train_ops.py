"""Train-mode encoder as a torch.autograd.Function over the C ABI (lrn_encoder_train_forward/backward).

Autograd only sees one node: inputs = the 28 encoder parameters (+ the context, which gets no gradient),
output = `fused` (B,1024,N).  Pooling and context_proj stay ordinary differentiable torch ops of `fused`,
so DDP's gradient hooks fire on the leaf parameters exactly as with the reference module
(reference train_dist.py:147,188)."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import lib
from .ops import _aligned_bytes, _call, _f32c

# parameter order of the autograd node (names relative to MultiScalePointNetEncoder)
PARAM_NAMES = ([f"conv{k}.weight" for k in range(1, 6)] + [f"conv{k}.bias" for k in range(1, 6)]
               + [f"bn{k}.weight" for k in range(1, 6)] + [f"bn{k}.bias" for k in range(1, 6)]
               + ["fusion.0.weight", "fusion.0.bias", "fusion.1.weight", "fusion.1.bias",
                  "intensity_gate.0.weight", "intensity_gate.0.bias", "intensity_gate.2.weight", "intensity_gate.2.bias"])


def _params_struct(t, eps=1e-5):
    """t: list of contiguous fp32 CUDA tensors in PARAM_NAMES order; eps: the BatchNorm layers' eps."""
    p = _lib.EncoderParams()
    for k in range(5):
        p.conv_w[k], p.conv_b[k] = t[k].data_ptr(), t[5 + k].data_ptr()
        p.bn_w[k], p.bn_b[k] = t[10 + k].data_ptr(), t[15 + k].data_ptr()
    p.fusion_w, p.fusion_b, p.fusion_bn_w, p.fusion_bn_b = (x.data_ptr() for x in t[20:24])
    p.gate0_w, p.gate0_b, p.gate2_w, p.gate2_b = (x.data_ptr() for x in t[24:28])
    p.bn_eps = float(eps)
    return p


class EncoderTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, context, running, momentum, eps, point_major, *params):
        """context (B,N,4) fp32 CUDA; running = list of 12 buffers (6 running_mean, 6 running_var) updated in
        place, or None; params in PARAM_NAMES order.  Returns (global_feat (B,2048), fused (B,1024,N)) fp32, or with
        point_major the (B,N,1024) bf16 tensor context_proj consumes (LineRefineNet never uses global_feat)."""
        context = _f32c(context)
        B, N, _ = context.shape
        dev = context.device
        t = [_f32c(p.detach()) for p in params]
        ps = _params_struct(t, eps)
        nbytes = lib.lrn_train_workspace_bytes(B, N)
        ws = _aligned_bytes(nbytes, dev)           # owned by this node until its backward has run
        fused = (torch.empty(B, N, 1024, dtype=torch.bfloat16, device=dev) if point_major
                 else torch.empty(B, 1024, N, dtype=torch.float32, device=dev))
        gf = am = None
        if not point_major:
            gf = torch.empty(B, 2048, dtype=torch.float32, device=dev)
            am = torch.empty(B, 1024, dtype=torch.int64, device=dev)
        rs = None
        if running is not None:
            rs = _lib.BnRunning()
            for i in range(6):
                rs.mean[i], rs.var[i] = running[i].data_ptr(), running[6 + i].data_ptr()
        _call("lrn_encoder_train_forward", dev, C.byref(ps), C.byref(rs) if rs is not None else None, momentum, context, B, N,
              fused, int(point_major), gf, am, ws, ws.numel())
        ctx.save_for_backward(context, *t)
        ctx.ws, ctx.shape, ctx.point_major, ctx.argmax, ctx.eps = ws, (B, N), bool(point_major), am, float(eps)
        if point_major:
            return fused
        ctx.mark_non_differentiable(am)
        return gf, fused, am

    @staticmethod
    def backward(ctx, *douts):
        context, *t = ctx.saved_tensors
        B, N = ctx.shape
        dev = context.device
        if ctx.ws is None:
            raise RuntimeError("pointnet_refine_b200: the native encoder's saved activations (12 KB per point) are released "
                               "by its first backward; a second backward through the same forward (retain_graph=True) is "
                               "not supported -- run the forward again")
        if ctx.point_major:
            d_gf, d_fused = None, douts[0].to(torch.bfloat16).contiguous()
        else:
            d_gf = _f32c(douts[0]) if douts[0] is not None else None
            d_fused = _f32c(douts[1]) if douts[1] is not None else None
        grads = [torch.empty_like(x) for x in t]
        g = _lib.EncoderGrads()
        for k in range(5):
            g.conv_w[k], g.conv_b[k] = grads[k].data_ptr(), grads[5 + k].data_ptr()
            g.bn_w[k], g.bn_b[k] = grads[10 + k].data_ptr(), grads[15 + k].data_ptr()
        g.fusion_w, g.fusion_b, g.fusion_bn_w, g.fusion_bn_b = (x.data_ptr() for x in grads[20:24])
        g.gate0_w, g.gate0_b, g.gate2_w, g.gate2_b = (x.data_ptr() for x in grads[24:28])
        ps = _params_struct(t, ctx.eps)
        _call("lrn_encoder_train_backward", dev, C.byref(ps), context, B, N, d_fused, int(ctx.point_major), d_gf,
              ctx.argmax if d_gf is not None else None, C.byref(g), ctx.ws, ctx.ws.numel())
        ctx.ws = None
        return (None, None, None, None, None, *grads)


def _encoder_bns(module):
    return [module.bn1, module.bn2, module.bn3, module.bn4, module.bn5, module.fusion[1]]


def native_train_supported(module) -> bool:
    """Whether the encoder `module` trains on the native path: it is in train mode, opted in (`native_training`), in the
    bf16 tier, and its BatchNorms behave as torch.nn.BatchNorm1d does by default in training, which is what the native
    path implements: every one in training mode with running statistics, an exponential momentum and one common eps.
    Anything else (frozen / .eval()'d BatchNorm layers, momentum=None cumulative averaging, track_running_stats=False)
    runs the stock ops."""
    if not (module.training and module.native_training and module.precision == "bf16"):
        return False
    bns = _encoder_bns(module)
    return all(b.training and b.track_running_stats and b.momentum is not None and b.affine and b.eps == bns[0].eps
               and b.momentum == bns[0].momentum for b in bns)


def encoder_train_forward(module, context, point_major=False):
    """module: MultiScalePointNetEncoder in train mode; context (B,N,4).  Returns (global_feat, fused) with
    autograd through the native backward; updates running statistics / num_batches_tracked like PyTorch.
    point_major=True returns (None, fused_pm (B,N,1024) bf16) for LineRefineNet, which never uses global_feat."""
    sd = dict(module.named_parameters())
    params = [sd[n] for n in PARAM_NAMES]
    bns = _encoder_bns(module)
    running = [b.running_mean for b in bns] + [b.running_var for b in bns]
    out = EncoderTrainFn.apply(context, running, float(bns[0].momentum), float(bns[0].eps), point_major, *params)
    with torch.no_grad():
        for b in bns:
            b.num_batches_tracked += 1
    if point_major:
        return None, out
    global_feat, fused, _ = out      # pooling (src/model.py:58-60) and its argmax-scatter backward are native too
    return global_feat, fused


def _col_sum(dyb):
    """Column sums (fp32) of a contiguous bf16 matrix: the bias gradient."""
    rows, cols = dyb.shape
    if cols % 64:
        return dyb.sum(dim=0, dtype=torch.float32)
    out = torch.empty(cols, dtype=torch.float32, device=dyb.device)
    _call("lrn_col_sum_bf16", dyb.device, dyb, dyb.stride(0), rows, cols, out)
    return out


class LinearBf16Fn(torch.autograd.Function):
    """y = x W^T + b on the tcgen05 GEMMs with bf16 operands and fp32 parameters / gradients:
    forward `lrn_gemm_bias_act`, dgrad `dy W` (K-major GEMM on W^T), wgrad `dy^T x` (`lrn_gemm_tn`, MN-major operands,
    split-K).  x (P, K) any float dtype, W (N, K) fp32, b (N) fp32; K % 64 == 0, N % 128 == 0.  Output bf16."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_dtype=torch.bfloat16):
        from . import ops
        xb = x.detach().to(torch.bfloat16).contiguous()
        wb = weight.detach().to(torch.bfloat16).contiguous()
        ctx.save_for_backward(xb, wb)
        ctx.needs = (x.requires_grad, weight.requires_grad, bias is not None and bias.requires_grad)
        ctx.x_dtype = x.dtype
        return ops.gemm_bias_act(xb, wb, bias.detach() if bias is not None else None, out_dtype=out_dtype)

    @staticmethod
    def backward(ctx, dy):
        from . import ops
        xb, wb = ctx.saved_tensors
        dyb = dy.to(torch.bfloat16).contiguous()
        need_x, need_w, need_b = ctx.needs
        dx = dw = db = None
        if need_x:
            direct = ctx.x_dtype in (torch.float32, torch.bfloat16)     # fp32 straight from the accumulators: no cast pass
            dx = ops.gemm_bias_act(dyb, wb.t().contiguous(), None, out_dtype=ctx.x_dtype if direct else torch.bfloat16)
            if not direct:
                dx = dx.to(ctx.x_dtype)
        if need_w:
            dw = ops.gemm_tn(dyb, xb)
        if need_b:
            db = _col_sum(dyb)
        return dx, dw, db, None


class KVGradShare:
    """One per training forward: the two (B, N, L, H, 32) bf16 buffers into which every layer's cross-attention backward
    (CrossAttnTrainFn) writes dK / dV in place; the K / V projections' backward then reads them as they are."""

    def __init__(self):
        self.dk = self.dv = None

    def buffers(self, B, N, L, device):
        if self.dk is None:
            self.dk = torch.empty(B, N, L, 8, 32, dtype=torch.bfloat16, device=device)
            self.dv = torch.empty_like(self.dk)
        return self.dk, self.dv


class KVProjFn(torch.autograd.Function):
    """K (or V) projections of all L cross-attention layers as ONE bf16 tensor-core linear over the context points,
    handed to the attention as L views (B, H, N, hd) of the (B, N, L, H, hd) result.  The backward reads the L attention
    gradients from the matching KVGradShare buffer (dK for the K projection, dV for V), where CrossAttnTrainFn wrote
    them in place, then dgrad / wgrad run like LinearBf16Fn.  x (B, N, K) bf16 or fp32, weight (L*H*hd, K) fp32,
    bias fp32."""

    @staticmethod
    def forward(ctx, x, weight, bias, L, H, share, key):
        from . import ops
        B, N, K = x.shape
        ctx.key = bool(key)
        xb = x.detach().to(torch.bfloat16).contiguous().view(B * N, K)
        wb = weight.detach().to(torch.bfloat16).contiguous()
        ctx.save_for_backward(xb, wb)
        ctx.needs = (x.requires_grad, weight.requires_grad, bias.requires_grad)
        ctx.meta = (B, N, K, L, H, x.dtype)
        ctx.share = share
        y = ops.gemm_bias_act(xb, wb, bias.detach(), out_dtype=torch.bfloat16).view(B, N, L, H, -1)
        return tuple(y[:, :, i].transpose(1, 2) for i in range(L))

    @staticmethod
    def backward(ctx, *grads):
        from . import ops
        xb, wb = ctx.saved_tensors
        B, N, K, L, H, x_dtype = ctx.meta
        dk, dv = ctx.share.buffers(B, N, L, xb.device)
        dy = dk if ctx.key else dv
        for i, g in enumerate(grads):
            block = dy[:, :, i]
            if g.data_ptr() != block.data_ptr():
                # autograd materialised this gradient (zeros): the layer's output is not on the loss's graph, so its
                # attention backward never wrote the block
                block.copy_(g.transpose(1, 2))
        dyb = dy.view(B * N, -1)
        need_x, need_w, need_b = ctx.needs
        dx = dw = db = None
        if need_x:
            dx = ops.gemm_bias_act(dyb, wb.t().contiguous(), None, out_dtype=torch.bfloat16).view(B, N, K).to(x_dtype)
        if need_w:
            dw = ops.gemm_tn(dyb, xb)
        if need_b:
            # K projection: a key bias shifts every score of a query by the same amount, which softmax ignores, so its
            # gradient sum_n dK[n] vanishes identically (rows of the score gradient sum to zero, with or without dropout);
            # the reference produces fp32 rounding noise there, a bf16 column sum would produce more - write the exact zero
            db = torch.zeros(wb.shape[0], dtype=torch.float32, device=xb.device) if ctx.key else _col_sum(dyb)
        return dx, dw, db, None, None, None, None


def kv_proj(x, weight, bias, layers: int, heads: int, share: KVGradShare, key: bool):
    """(B, N, K) -> tuple of `layers` tensors (B, heads, N, hd), see KVProjFn.  key: the K projection (its gradients
    come from share.dk and its bias gradient is identically zero), else the V projection (share.dv)."""
    return KVProjFn.apply(x, weight, bias, layers, heads, share, key)


class DropoutSeedState:
    """Where the train attention kernels' dropout seed comes from.  Default: a fresh 62-bit draw from torch's host
    generator per attention call, passed as a launch argument.  Under a CUDA-graph capture launch arguments are frozen,
    so graph.GraphedTrainStep installs a device word here instead (`word`, int64 on the GPU, advanced inside the
    graph): every attention call of the step then passes a fixed per-call salt as `seed` and the kernels add the word."""
    word = None      # int64 CUDA tensor of one element, or None
    calls = 0        # attention calls since the word was installed / the step began (the per-call salt)

    @classmethod
    def next(cls, p_drop):
        """(seed, seed_state pointer or None) for one attention call."""
        if p_drop <= 0:
            return 0, None
        if cls.word is None:
            return int(torch.randint(0, 2 ** 62, (1,)).item()), None     # host generator: follows torch.manual_seed
        cls.calls += 1
        return (cls.calls * 0x9E3779B97F4A7C15) & (2 ** 62 - 1), cls.word.data_ptr()


class CrossAttnTrainFn(torch.autograd.Function):
    """Attention of the 32 polyline queries of a segment in train mode (8 heads x 32, dropout on the attention weights),
    forward and backward on lrn_train_attention_*.  Cross attention: K / V are read straight from the K / V projection's
    (B, N, L, H, 32) buffer and dK / dV are written into the matching KVGradShare buffers in place.  Self attention:
    N = 32 keys, any row pitch.  q (B, 32, 256) fp32; k, v: (B, H, N, 32) bf16 views whose heads are 32 elements apart."""

    @staticmethod
    def forward(ctx, q, k, v, p_drop, share, layer):
        q = _f32c(q.detach())
        B, H, N, hd = k.shape
        ldk, ldv = k.stride(2), v.stride(2)
        if (H, hd) != (8, 32) or tuple(q.shape) != (B, 32, 256) or k.dtype != torch.bfloat16 or v.dtype != torch.bfloat16 or \
                tuple(k.stride()) != (N * ldk, 32, ldk, 1) or tuple(v.stride()) != (N * ldv, 32, ldv, 1) or v.shape != k.shape:
            raise ValueError("CrossAttnTrainFn: expected q (B,32,256) and (B,8,N,32) bf16 views with heads 32 elements apart")
        out = torch.empty_like(q)
        lse = torch.empty(B, 8, 32, dtype=torch.float32, device=q.device)
        seed, seed_state = DropoutSeedState.next(p_drop)
        _call("lrn_train_attention_forward", q.device, q, k, ldk, v, ldv, B, N, out, lse, float(p_drop), seed, seed_state)
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.cfg = (float(p_drop), seed, seed_state, share, int(layer))
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, out, lse = ctx.saved_tensors
        p_drop, seed, seed_state, share, layer = ctx.cfg
        B, H, N, hd = k.shape
        dout = _f32c(dout)
        dq = torch.empty_like(q)
        L = k.stride(2) // (H * hd)                   # cross attention: k is the layer's column block of a (B, N, L, H, hd) buffer
        if share is not None and k.stride(2) == L * H * hd and v.stride(2) == k.stride(2) and layer < L:
            dk_all, dv_all = share.buffers(B, N, L, q.device)
            gk, gv = dk_all[:, :, layer].transpose(1, 2), dv_all[:, :, layer].transpose(1, 2)
        else:
            gk = torch.empty(B, N, H, hd, dtype=torch.bfloat16, device=q.device).transpose(1, 2)
            gv = torch.empty(B, N, H, hd, dtype=torch.bfloat16, device=q.device).transpose(1, 2)
        _call("lrn_train_attention_backward", q.device, q, k, k.stride(2), v, v.stride(2), B, N, out, lse, dout, dq, gk,
              gk.stride(2), gv, gv.stride(2), p_drop, seed, seed_state)
        return dq, gk, gv, None, None, None


def cross_attention_train(q, k, v, p_drop: float, share: KVGradShare | None, layer: int):
    """(B, 32, 256) fp32 attention output (heads concatenated, before out_proj); see CrossAttnTrainFn."""
    return CrossAttnTrainFn.apply(q, k, v, p_drop, share, layer)


def self_attention_train(qk, v, p_drop: float):
    """Self attention among the 32 polyline points of every segment in train mode (src/model.py:113-117) on the same
    kernels: qk (B, 32, 512) = [q | k] in-projections, v (B, 32, 256) (any float dtype; bf16 is used as is) ->
    (B, 32, 256) fp32, heads concatenated."""
    B = qk.shape[0]
    qkb, vb = qk.to(torch.bfloat16), v.to(torch.bfloat16)
    heads = lambda t: t.unflatten(-1, (8, 32)).transpose(1, 2)          # (B, 32, 256) view -> (B, 8, 32, 32), heads 32 apart
    return CrossAttnTrainFn.apply(qk[..., :256].float(), heads(qkb[..., 256:]), heads(vb), p_drop, None, 0)


class PosHiddenFn(torch.autograd.Function):
    """relu(W1 xyz + b1) on the context points as bf16 (lrn_pos_hidden), with the parameter gradients from
    lrn_pos_hidden_backward; the context itself gets no gradient (PositionalEncoding.mlp[0], src/model.py:66-75,197)."""

    @staticmethod
    def forward(ctx, context, w1, b1):
        context = _f32c(context)
        B, N, _ = context.shape
        h = torch.empty(B, N, 256, dtype=torch.bfloat16, device=context.device)
        _call("lrn_pos_hidden", context.device, _f32c(w1.detach()), _f32c(b1.detach()), context, B * N, h, 256)
        ctx.save_for_backward(context, h)
        return h

    @staticmethod
    def backward(ctx, dh):
        context, h = ctx.saved_tensors
        dh = dh.to(torch.bfloat16).contiguous()
        dw = torch.empty(256, 3, dtype=torch.float32, device=h.device)
        db = torch.empty(256, dtype=torch.float32, device=h.device)
        _call("lrn_pos_hidden_backward", h.device, context, h.numel() // 256, h, 256, dh, 256, dw, db)
        return None, dw, db


def pos_hidden_train(context, w1, b1):
    return PosHiddenFn.apply(context, w1, b1)


class AddLayerNormFn(torch.autograd.Function):
    """LayerNorm(x + y) over 256 columns with the residual add fused in, forward and backward on the native kernels
    (lrn_add_layernorm / lrn_add_layernorm_backward); norm1 / norm2 / norm3 of DetrTransformerDecoderLayer in training."""

    @staticmethod
    def forward(ctx, x, y, gamma, beta, eps):
        x, y = _f32c(x), _f32c(y)
        g, b = _f32c(gamma.detach()), _f32c(beta.detach())
        rows = x.numel() // 256
        out = torch.empty_like(x)
        stats = torch.empty(rows, 2, dtype=torch.float32, device=x.device)
        _call("lrn_add_layernorm", x.device, x, y, g, b, float(eps), out, stats, rows, 256)
        ctx.save_for_backward(x, y, stats, g)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, y, stats, g = ctx.saved_tensors
        dout = _f32c(dout)
        dz = torch.empty_like(x)
        dgamma = torch.empty(256, dtype=torch.float32, device=x.device)
        dbeta = torch.empty(256, dtype=torch.float32, device=x.device)
        _call("lrn_add_layernorm_backward", x.device, dout, x, y, stats, g, dz, dgamma, dbeta, x.numel() // 256, 256)
        return dz, dz, dgamma, dbeta, None


def add_layernorm(x, y, norm: torch.nn.LayerNorm):
    """norm(x + y), differentiable, for (..., 256) fp32 CUDA tensors."""
    if x.shape[-1] != 256 or x.shape != y.shape:
        raise ValueError(f"add_layernorm: shapes {tuple(x.shape)}, {tuple(y.shape)} (last dim must be 256)")
    return AddLayerNormFn.apply(x, y, norm.weight, norm.bias, norm.eps)


class ThinLinearFn(torch.autograd.Function):
    """fp32 y = x W^T + b for the layers with 3 input or 3 output features on the polyline rows (pos_emb.mlp[0] on the
    current points, reg_branches[i][2]; src/model.py:66-75,172-179).  Forward and dx are ordinary small matmuls; the weight
    gradient dW = dy^T x reduces over ALL rows (32 k at B = 1024) into a 256 x 3 or 3 x 128 result, which a library GEMM
    runs as one or two CTAs looping over K (80 us per launch, 12 per step): here the rows are split into 64 slabs whose
    partial products come from one batched matmul and are summed (two launches of a few microseconds)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        return torch.nn.functional.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dx = dw = db = None
        dy2 = dy.reshape(-1, dy.shape[-1])
        x2 = x.reshape(-1, x.shape[-1])
        if ctx.needs_input_grad[0]:
            dx = (dy2 @ weight).view(x.shape)
        if ctx.needs_input_grad[1]:
            rows = dy2.shape[0]
            slabs = 64 if rows % 64 == 0 and rows >= 4096 else 1
            if slabs > 1:
                dw = torch.bmm(dy2.view(slabs, rows // slabs, -1).transpose(1, 2), x2.view(slabs, rows // slabs, -1)).sum(0)
            else:
                dw = dy2.t() @ x2
        if ctx.needs_input_grad[2]:
            db = dy2.sum(0)
        return dx, dw, db


def thin_linear(x, weight, bias):
    return ThinLinearFn.apply(x, weight, bias)


def linear_bf16(x, weight, bias, out_dtype=torch.bfloat16):
    """Differentiable bf16 tensor-core linear layer over the last dimension of x (leading dims flattened); the result is
    bf16, or fp32 written straight from the accumulators (out_dtype=torch.float32: no conversion pass for consumers that
    want fp32, e.g. the residual + LayerNorm kernels)."""
    lead = x.shape[:-1]
    y = LinearBf16Fn.apply(x.reshape(-1, x.shape[-1]), weight, bias, out_dtype)
    return y.view(*lead, weight.shape[0])
