"""Host-side mirror of the reference's module interface (reference: src/model.py).

Same class names, constructor arguments, parameter/buffer tree (205 state_dict keys, SURVEY.md
appendix B) and forward signatures as the reference, so ``load_state_dict(strict=True)`` of a
reference checkpoint works and ``train.py`` / ``inference*.py`` run unchanged with
``from src.model import LineRefineNet`` resolved to this file (see compat/src/model.py).

What runs where
  * eval mode, CUDA tensors: the context encoder (+ pooling, + context_proj) and the regression
    heads run in the hand-written sm_100a library through the C ABI (ops.py).  In the bf16 and tf32 tiers
    with M = 32 polyline points the whole decoder does too (LineRefineNet._refine_native); the fp32x3 tier
    and M != 32 run the DETR decoder and pos_emb in stock fp32 PyTorch ops (LineRefineNet._refine).
  * train mode (batch-statistic BatchNorm, autograd): by default the stock PyTorch fp32 formulation, i.e. exactly
    the reference's numerics (a bf16 forward flips the ReLU mask of a few per mille of the activations, which is
    within tolerance for inference but changes gradients -- the caller decides).  `native_training = True` /
    LRN_NATIVE_TRAIN=1 (bf16 tier) switches the encoder, and with M = 32 also context_proj and the decoder's linears and
    attention, to the sm_100a train path (train_ops.py: batch-stat BN forward and a hand-written backward on the tcgen05
    GEMMs).
  * CPU tensors: not supported -- there is no CPU path in the product (the oracle lives in oracle/).
"""
from __future__ import annotations

import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, train_ops

_DEFAULT_PRECISION = os.environ.get("LRN_PRECISION", "bf16")


_warned_autograd = False


def _use_native(module: nn.Module, *inputs) -> bool:
    """The sm_100a kernels implement the eval-mode forward without autograd.  Train mode, or an
    eval-mode call that autograd is recording, runs the stock-PyTorch formulation instead (and says
    so once): inference scripts call ``model.eval()`` under ``torch.no_grad()`` (reference
    inference_whole_scene.py:134-137) and always take the native path."""
    global _warned_autograd
    if module.training:
        return False
    if torch.is_grad_enabled() and (any(t.requires_grad for t in inputs)
                                    or any(p.requires_grad for p in module.parameters())):
        if not _warned_autograd:
            import warnings
            warnings.warn("pointnet_refine_b200: eval-mode forward is being recorded by autograd; using the "
                          "stock PyTorch formulation. Wrap inference in torch.no_grad() for the sm_100a path.")
            _warned_autograd = True
        return False
    return True


def _require_cuda(t: torch.Tensor, who: str):
    if not t.is_cuda:
        raise RuntimeError(f"{who}: the B200-native path has no CPU implementation; move the module and "
                           f"its inputs to a CUDA device (sm_100a).")


def _prepared(cache: dict, name, sources, build, key=()):
    """cache[name], a weight prepared from parameters (BN fold, re-packed or rounded copy): build() is called again when
    the (data_ptr, _version) fingerprint of `sources` or the extra `key` changes.  That catches optimizer steps,
    load_state_dict and .to(); an in-place edit through `.data` bumps no version, hence the modules' invalidate()."""
    fp = key + tuple((t.data_ptr(), t._version) for t in sources)
    hit = cache.get(name)
    if hit is None or hit[0] != fp:
        cache[name] = hit = (fp, build())
    return hit[1]


class MultiScalePointNetEncoder(nn.Module):
    """Per-point shared MLP 4->64->128->256->512->1024, multi-scale fusion 1984->1024, intensity
    gate, max+avg pooling.  Interface of reference src/model.py:5-62:
    ``forward(x: (B,4,N)) -> (global_feat (B,2048), fused (B,1024,N))``."""

    def __init__(self, in_channel=4, out_dim=1024):
        super().__init__()
        if in_channel != 4 or out_dim != 1024:
            raise ValueError("the sm_100a kernels are specialised for in_channel=4, out_dim=1024 "
                             "(the only configuration the reference instantiates, src/model.py:146)")
        widths = (in_channel, 64, 128, 256, 512, out_dim)
        for k in range(1, 6):
            setattr(self, f"conv{k}", nn.Conv1d(widths[k - 1], widths[k], 1))
        for k in range(1, 6):
            setattr(self, f"bn{k}", nn.BatchNorm1d(widths[k]))
        self.fusion = nn.Sequential(nn.Conv1d(sum(widths[1:]), out_dim, 1), nn.BatchNorm1d(out_dim), nn.ReLU())
        self.intensity_gate = nn.Sequential(nn.Conv1d(1, 64, 1), nn.ReLU(), nn.Conv1d(64, out_dim, 1), nn.Sigmoid())
        self.precision = _DEFAULT_PRECISION     # "bf16" | "tf32" | "fp32x3" (tensor-core operand tier; fp32x3 = 3 x TF32 split, fp32-class)
        self.chunk_rows = 0                     # 0 = library default
        self.native_training = os.environ.get("LRN_NATIVE_TRAIN", "0") == "1"   # opt-in: train mode on the sm_100a kernels (bf16)
        self._prepared = {}                     # prepared weights (_prepared); never in the state_dict
        self._proj = None                       # optional nn.Linear(1024,256) folded alongside (set by LineRefineNet)

    def folded(self) -> ops.FoldedEncoder:
        """BN-folded operand blob for the current parameters; re-folded whenever a parameter or
        running statistic changes (optimizer step, load_state_dict, .to())."""
        ts = list(self.parameters()) + list(self.buffers())
        if self._proj is not None:
            ts += list(self._proj[0].parameters())

        def fold():
            tensors = {k: v for k, v in self.state_dict().items() if v.is_floating_point()}
            if self._proj is not None:
                tensors["context_proj.weight"] = self._proj[0].weight
                tensors["context_proj.bias"] = self._proj[0].bias
            return ops.FoldedEncoder(tensors, self.precision, bn_eps=self.bn1.eps)
        return _prepared(self._prepared, "fold", ts, fold, key=(self.precision,))

    def invalidate(self):
        """Drop the prepared weights.  They are keyed on (data_ptr, _version) of every parameter and buffer, which
        catches optimizer steps, load_state_dict and .to(); an in-place edit THROUGH `.data` (p.data.copy_(ema),
        p.data.mul_(...)) does not bump `_version` - call this (or LineRefineNet.invalidate()) after such an edit."""
        self._prepared.clear()

    # -- forward ---------------------------------------------------------------------------------
    def run_native(self, context, **outputs):
        """context (B,N,4) -> dict of requested outputs (see ops.encoder_forward)."""
        _require_cuda(context, "MultiScalePointNetEncoder")
        return ops.encoder_forward(self.folded(), context, chunk_rows=self.chunk_rows, **outputs)

    def _forward_torch(self, x):
        """Autograd-capable forward with stock PyTorch ops (batch-statistic BN in train mode)."""
        feats, h = [], x
        for k in range(1, 6):
            h = F.relu(getattr(self, f"bn{k}")(getattr(self, f"conv{k}")(h)))
            feats.append(h)
        fused = self.fusion(torch.cat(feats, dim=1)) * (0.5 + 0.5 * self.intensity_gate(x[:, 3:4, :]))
        return torch.cat([fused.max(dim=2)[0], fused.mean(dim=2)], dim=1), fused

    def forward(self, x):
        _require_cuda(x, "MultiScalePointNetEncoder")
        if train_ops.native_train_supported(self):   # batch-stat BN forward + hand-written backward
            return train_ops.encoder_train_forward(self, x.transpose(2, 1))
        if not _use_native(self, x):
            return self._forward_torch(x)
        out = self.run_native(x.transpose(2, 1), pool=True, fused=True)
        return out["global_feat"], out["fused"]


class PositionalEncoding(nn.Module):
    """MLP positional encoding 3->256->256 (reference src/model.py:64-75)."""

    def __init__(self, in_dim=3, out_dim=256):
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(in_dim, out_dim), nn.ReLU(), nn.Linear(out_dim, out_dim))

    def forward(self, xyz):
        return self.mlp(xyz)


class DetrTransformerDecoderLayer(nn.Module):
    """Post-norm DETR decoder layer (reference src/model.py:77-135): self-attention over the line
    queries, cross-attention into the context memory, FFN.  Stock PyTorch ops (section 8f row 1-2)."""

    def __init__(self, d_model=256, nhead=8, dim_feedforward=1024, dropout=0.1):
        super().__init__()
        self.self_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout, batch_first=True)
        self.cross_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout, batch_first=True)
        self.linear1 = nn.Linear(d_model, dim_feedforward)
        self.dropout = nn.Dropout(dropout)
        self.linear2 = nn.Linear(dim_feedforward, d_model)
        self.norm1, self.norm2, self.norm3 = (nn.LayerNorm(d_model) for _ in range(3))
        self.dropout1, self.dropout2, self.dropout3 = (nn.Dropout(dropout) for _ in range(3))
        self.activation = F.relu

    @staticmethod
    def with_pos_embed(tensor, pos):
        return tensor if pos is None else tensor + pos

    def forward(self, tgt, memory, query_pos=None, pos=None):
        q = self.with_pos_embed(tgt, query_pos)
        tgt = self.norm1(tgt + self.dropout1(self.self_attn(q, q, value=tgt, need_weights=False)[0]))
        attn = self.cross_attn(self.with_pos_embed(tgt, query_pos), self.with_pos_embed(memory, pos), value=memory,
                               need_weights=False)[0]
        tgt = self.norm2(tgt + self.dropout2(attn))
        ffn = self.linear2(self.dropout(self.activation(self.linear1(tgt))))
        return self.norm3(tgt + self.dropout3(ffn))


class LineRefineNet(nn.Module):
    """Reference src/model.py:137-234.  forward(context (B,N,4), noisy_line (B,M,3)) -> (6,B,M,3)
    cumulative offsets per decoder layer."""

    def __init__(self, num_line_points=32, feature_dim=1024):
        super().__init__()
        self.d_model = 256
        self.num_decoder_layers = 6
        self.context_encoder = MultiScalePointNetEncoder(in_channel=4, out_dim=feature_dim)
        self.context_proj = nn.Linear(feature_dim, self.d_model)
        self.point_mlp = nn.Sequential(
            nn.Conv1d(3, 64, 1), nn.BatchNorm1d(64), nn.ReLU(),
            nn.Conv1d(64, 128, 1), nn.BatchNorm1d(128), nn.ReLU(),
            nn.Conv1d(128, self.d_model, 1), nn.BatchNorm1d(self.d_model))
        self.pos_emb = PositionalEncoding(in_dim=3, out_dim=self.d_model)
        self.decoder_layers = nn.ModuleList(
            [DetrTransformerDecoderLayer(self.d_model, 8, 1024) for _ in range(self.num_decoder_layers)])
        self.reg_branches = nn.ModuleList(
            [nn.Sequential(nn.Linear(self.d_model, 128), nn.ReLU(), nn.Linear(128, 3))
             for _ in range(self.num_decoder_layers)])
        # context_proj is folded into the encoder's operand blob (tuple hides it from the module tree)
        self.context_encoder._proj = (self.context_proj,)
        self._prepared = self.context_encoder._prepared   # one cache for the encoder fold and the decoder's prepared weights
        self.segment_chunk = 256   # segments per decoder pass in eval mode (bounds the (B,N,256) temporaries)

    def invalidate(self):
        """Drop every prepared weight (encoder fold, folded attention weights, point_mlp fold, K / V copies, TF32
        copies): needed only after in-place parameter edits through `.data`, which the (data_ptr, _version) fingerprints
        cannot see; optimizer steps, load_state_dict and .to() are detected automatically."""
        self._prepared.clear()

    @property
    def precision(self):
        return self.context_encoder.precision

    @precision.setter
    def precision(self, value):
        self.context_encoder.precision = value

    def _refine(self, context, noisy_line, memory, native_heads):
        pos_mem = self.pos_emb(context[:, :, :3])
        if native_heads:   # eval: point_mlp with its BatchNorms folded, fp32 FMA (cuDNN would run the 1x1 convs in TF32 by default)
            (pw1, pb1), (pw2, pb2), (pw3, pb3) = self._point_mlp_weights()
            tgt = ops.rows_linear(ops.rows_linear(noisy_line, pw2, pb2, mlp3=(pw1, pb1), relu=True), pw3, pb3)
        else:
            tgt = self.point_mlp(noisy_line.transpose(2, 1)).transpose(2, 1)
        current = noisy_line.clone()
        outs = []
        for layer, head in zip(self.decoder_layers, self.reg_branches):
            tgt = layer(tgt, memory, query_pos=self.pos_emb(current), pos=pos_mem)
            if native_heads:
                outs.append(ops.head_forward(head[0].weight, head[0].bias, head[2].weight, head[2].bias,
                                             tgt, current, noisy_line))
            else:
                current = current + head(tgt)
                outs.append(current - noisy_line)
        return torch.stack(outs)

    # -- context side of the decoder on the tcgen05 GEMMs (SURVEY.md section 8f row 1) ------------------------
    @staticmethod
    def _rna_tf32(t):
        """fp32 -> nearest TF32 value (ties away from zero in magnitude), still stored as fp32: the tensor core would
        otherwise truncate the low 13 mantissa bits of every operand, a bias that adds up over K."""
        return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)

    def _kv_weights(self):
        """Copies, rounded to the nearest TF32 value, of pos_emb.mlp.2 and of the K / V rows of all six cross-attention
        in_proj matrices ([Wq; Wk; Wv] packing of nn.MultiheadAttention), re-made when a parameter changes: the operands
        of the tf32 tier's context-side GEMMs.  Host-side weight preparation (like _attn_weights)."""
        ps = [self.pos_emb.mlp[2].weight, self.pos_emb.mlp[2].bias]
        for l in self.decoder_layers:
            ps += [l.cross_attn.in_proj_weight, l.cross_attn.in_proj_bias]

        def build():
            d = self.d_model
            dev = ps[0].device
            host = lambda t: t.detach().cpu().float()
            wk = torch.cat([host(l.cross_attn.in_proj_weight)[d:2 * d] for l in self.decoder_layers])
            wv = torch.cat([host(l.cross_attn.in_proj_weight)[2 * d:] for l in self.decoder_layers])
            bk = torch.cat([host(l.cross_attn.in_proj_bias)[d:2 * d] for l in self.decoder_layers])
            bv = torch.cat([host(l.cross_attn.in_proj_bias)[2 * d:] for l in self.decoder_layers])
            cast = lambda t: self._rna_tf32(t).to(dev)
            return (cast(wk), bk.contiguous().to(dev), cast(wv), bv.contiguous().to(dev), cast(host(self.pos_emb.mlp[2].weight)))
        return _prepared(self._prepared, "kv", ps, build)

    def _tf32_weight(self, w):
        """fp32 weight (or a row slice of one) rounded to the nearest TF32 value, cached until the parameter changes:
        the operand form of the tf32 tier's tensor-core linears (native rounding kernel, once per parameter update)."""
        return _prepared(self._prepared, ("tf32", w.data_ptr()), [w], lambda: ops.add(w.detach(), None, round_tf32=True),
                         key=tuple(w.shape))

    # -- cross attention without K / V: folded queries + lrn_ctx_attention ------------------------------------
    def _attn_weights(self):
        """Per cross-attention layer, the query and output sides with the K / V projections folded in
        (csrc/ctx_attn_sm100.cuh):  Wqk (2048,256), bqk: (tgt+qpos) -> 8 heads x 256 folded query (scores come out
        in log2 units, 1/sqrt(32) included);  Wvo (256,2048), bvo: 8 heads x (softmax . memory) -> out_proj output.
        Plus [I | pos_emb.mlp.2.weight] (256,512) bf16, so that one GEMM over [memory | pos hidden] rows gives
        memory + pos.  Weight preparation, not data path: computed on the host in float64 once per parameter change
        (like lrn_encoder_fold, it must be redone when a parameter changes) and uploaded."""
        ps = [self.pos_emb.mlp[2].weight, self.pos_emb.mlp[2].bias]
        for l in self.decoder_layers:
            ps += [l.cross_attn.in_proj_weight, l.cross_attn.in_proj_bias, l.cross_attn.out_proj.weight, l.cross_attn.out_proj.bias]

        def build():
            d, H = self.d_model, 8
            hd = d // H
            dev = ps[0].device
            scale = math.log2(math.e) / math.sqrt(hd)
            host = lambda t: t.detach().cpu().double()
            up = lambda t, dt=torch.float32: t.to(dt).contiguous().to(dev)
            layers = []
            for l in self.decoder_layers:
                ca = l.cross_attn
                w, b = host(ca.in_proj_weight), host(ca.in_proj_bias)
                wq, wk, wv = w[:d].view(H, hd, d), w[d:2 * d].view(H, hd, d), w[2 * d:].view(H, hd, d)
                bq, bv = b[:d].view(H, hd), b[2 * d:]
                wo, bo = host(ca.out_proj.weight), host(ca.out_proj.bias)
                wqk = scale * torch.einsum("hcd,hce->hde", wk, wq).reshape(H * d, d)          # row h*256+j: folded dim j of head h
                bqk = scale * torch.einsum("hc,hcd->hd", bq, wk).reshape(H * d)
                wvo = torch.einsum("ohc,hcd->ohd", wo.view(d, H, hd), wv).reshape(d, H * d)
                bvo = wo @ bv + bo
                layers.append((up(wqk), up(bqk), up(wvo), up(bvo), up(wvo.float(), torch.bfloat16)))
            w2 = host(self.pos_emb.mlp[2].weight)
            wx = up(torch.cat([torch.eye(d, dtype=w2.dtype), w2], dim=1).float(), torch.bfloat16)
            return layers, wx, up(host(self.pos_emb.mlp[2].bias))
        return _prepared(self._prepared, "attn", ps, build)

    def _point_mlp_weights(self):
        """point_mlp (src/model.py:150-159) with its three eval-mode BatchNorms folded into the 1x1 convs:
        [(W1 (64,3), b1), (W2 (128,64), b2), (W3 (256,128), b3)] fp32.  Host-side weight preparation, cached like _attn_weights."""
        ts = list(self.point_mlp.parameters()) + list(self.point_mlp.buffers())

        def build():
            dev = ts[0].device
            out = []
            for ci, bi in ((0, 1), (3, 4), (6, 7)):
                conv, bn = self.point_mlp[ci], self.point_mlp[bi]
                s = bn.weight.detach().cpu().double() / torch.sqrt(bn.running_var.detach().cpu().double() + bn.eps)
                w = conv.weight.detach().cpu().double().squeeze(-1) * s[:, None]
                b = (conv.bias.detach().cpu().double() - bn.running_mean.detach().cpu().double()) * s + bn.bias.detach().cpu().double()
                out.append((w.float().contiguous().to(dev), b.float().contiguous().to(dev)))
            return out
        return _prepared(self._prepared, "point_mlp", ts, build)

    def _refine_native(self, context, noisy_line, memory, out):
        """Eval-mode decoder of the bf16 and tf32 tiers at M = 32, every step on this library's kernels.  The tier supplies
        the context side and each layer's cross attention (_bf16_cross_attention over the encoder's (B,N,512) bf16
        LRN_OUT_MEMORY_BF16 buffer, _tf32_cross_attention over the (B,N,256) fp32 memory) and the operand form of the
        tensor-core linears.  The query side is shared: its linears run on the tcgen05 GEMM in its tf32 mode from 256
        polyline rows on, and as fp32 rows_linear launches below that (B < 8: the whole-scene loop's B = 1,
        inference_whole_scene.py:130-139); self attention, residual + LayerNorm, heads and the cumulative offsets are the
        kernels of csrc/query_kernels.cuh.  The six cumulative offsets go straight into `out` (6,B,32,3).  Same parameters
        and math as DetrTransformerDecoderLayer.forward (src/model.py:104-135)."""
        B = context.shape[0]
        d = self.d_model
        bf16 = self.precision == "bf16"
        rows = B * noisy_line.shape[1]
        big = rows >= 256     # thousands of rows: tensor-core linears; else one fp32 rows_linear launch per nn.Linear

        def lin(x, w, b, relu=False, out_dtype=None, add=None):   # (B,32,K) fp32 [+ add] -> (B,32,N) fp32 (or out_dtype)
            if not big:
                return ops.rows_linear(x, w, b, add=add, relu=relu, out_dtype=out_dtype or torch.float32)
            if not bf16:   # tf32 tier: operands rounded to the nearest TF32 value (the bf16 tier lets the tensor core truncate)
                x, w = ops.add(x, add, round_tf32=True), self._tf32_weight(w)
            elif add is not None:
                x = ops.add(x, add)
            return ops.gemm_bias_act(x.reshape(rows, -1), w.detach(), b.detach(), relu=relu, out_dtype=out_dtype).view(B, -1, w.shape[0])

        if bf16:
            cross_attention = self._bf16_cross_attention(context, memory, lin, big)
        else:
            cross_attention = self._tf32_cross_attention(context, memory, lin)
        (pw1, pb1), (pw2, pb2), (pw3, pb3) = self._point_mlp_weights()
        pe0, pe2 = self.pos_emb.mlp[0], self.pos_emb.mlp[2]
        tgt = ops.rows_linear(ops.rows_linear(noisy_line, pw2, pb2, mlp3=(pw1, pb1), relu=True), pw3, pb3)   # point_mlp
        current = noisy_line.clone()
        for i, (layer, head) in enumerate(zip(self.decoder_layers, self.reg_branches)):
            if big:
                qpos = lin(ops.query_pos_hidden(pe0.weight, pe0.bias, current), pe2.weight, pe2.bias)
            else:
                qpos = ops.rows_linear(current, pe2.weight, pe2.bias, mlp3=(pe0.weight, pe0.bias))
            sa = layer.self_attn
            qk = lin(tgt, sa.in_proj_weight[:2 * d], sa.in_proj_bias[:2 * d], add=qpos)
            v = lin(tgt, sa.in_proj_weight[2 * d:], sa.in_proj_bias[2 * d:])
            tgt = ops.add_layernorm(tgt, lin(ops.self_attention32(qk, v), sa.out_proj.weight, sa.out_proj.bias), layer.norm1)
            tgt = ops.add_layernorm(tgt, cross_attention(i, tgt, qpos), layer.norm2)
            ffn = lin(lin(tgt, layer.linear1.weight, layer.linear1.bias, relu=True), layer.linear2.weight, layer.linear2.bias)
            tgt = ops.add_layernorm(tgt, ffn, layer.norm3)
            hid = lin(tgt, head[0].weight, head[0].bias, relu=True)
            ops.head_update(hid, head[2].weight, head[2].bias, current, noisy_line, out=out[i])

    def _bf16_cross_attention(self, context, memx, lin, big):
        """bf16 tier: per layer the cross attention is ONE lrn_ctx_attention launch over kp = memory + pos and memory (bf16),
        with Wk / Wv folded into the 32 x 8 queries and into out_proj (_attn_weights) - K and V of nn.MultiheadAttention
        (src/model.py:123-128) are never formed.  `memx` (B,N,512) bf16 is the encoder's LRN_OUT_MEMORY_BF16 buffer:
        [memory | room for the positional hidden layer].  Returns layer i's step (tgt, qpos) -> out_proj output."""
        B, N, _ = context.shape
        d, H = self.d_model, 8
        layers_w, wx, b2 = self._attn_weights()
        ops.pos_hidden(self.pos_emb.mlp[0].weight.detach(), self.pos_emb.mlp[0].bias.detach(), context, memx[:, :, d:])
        kp = ops.gemm_bias_act(memx.view(B * N, 2 * d), wx, b2, out_dtype=torch.bfloat16).view(B, N, d)
        mem = memx[:, :, :d]

        def cross_attention(i, tgt, qpos):
            wqk, bqk, wvo, bvo, wvo16 = layers_w[i]
            # folded queries: row q * 8 + h of the segment's 256 (any row order works, rows are independent)
            qf = lin(tgt, wqk, bqk, out_dtype=torch.bfloat16, add=qpos).view(B, H * 32, d)   # fp32 / tf32 accumulate, rounded once
            if big:   # attention output leaves the kernel as bf16, Wv / out_proj (folded) is a bf16 GEMM with fp32 output
                o = ops.ctx_attention(qf, kp, mem, out_dtype=torch.bfloat16).view(B * 32, H * d)
                return ops.gemm_bias_act(o, wvo16, bvo, out_dtype=torch.float32).view(B, 32, d)
            return ops.rows_linear(ops.ctx_attention(qf, kp, mem).view(B, 32, H * d), wvo, bvo)
        return cross_attention

    def _tf32_cross_attention(self, context, memory, lin):
        """tf32 tier: the context-side work is hoisted out of the layer loop.  The memory positional embedding and the K / V
        projections of ALL six cross-attention layers are three TF32 tensor-core GEMMs over the points (they do not depend
        on the decoder state, src/model.py:123-126; operands rounded to the nearest TF32 value where they are produced -
        the tensor core would truncate, a bias that adds up over K), and every layer's cross attention is one fp32
        lrn_cross_attention32 launch on its column block of those K / V.  Returns layer i's step (tgt, qpos) -> out_proj
        output."""
        B, N, _ = context.shape
        d = self.d_model
        wk, bk, wv, bv, w2 = self._kv_weights()
        pe0, pe2 = self.pos_emb.mlp[0], self.pos_emb.mlp[2]
        mem = memory.reshape(B * N, d)
        h = ops.query_pos_hidden(pe0.weight, pe0.bias, context, round_tf32=True).view(B * N, d)
        posm = ops.gemm_bias_act(h, w2, pe2.bias.detach())
        k_all = ops.gemm_bias_act(ops.add(mem, posm, round_tf32=True), wk, bk).view(B, N, 6 * d)
        v_all = ops.gemm_bias_act(ops.add(mem, None, round_tf32=True), wv, bv).view(B, N, 6 * d)
        del h, posm

        def cross_attention(i, tgt, qpos):
            ca = self.decoder_layers[i].cross_attn
            qh = lin(tgt, ca.in_proj_weight[:d], ca.in_proj_bias[:d], add=qpos)
            att = ops.cross_attention32(qh, k_all[:, :, i * d:(i + 1) * d], v_all[:, :, i * d:(i + 1) * d])
            return lin(att, ca.out_proj.weight, ca.out_proj.bias)
        return cross_attention

    def _refine_fast_train(self, context, noisy_line, fused_pm):
        """Autograd-capable decoder of model.train() on the native encoder, for M = 32 polyline points: context_proj, the
        memory positional embedding and the K / V projections of all six cross-attention layers run as differentiable bf16
        tensor-core linears (train_ops.linear_bf16 / kv_proj: tcgen05 forward, dgrad and wgrad); the self attention of
        the 32 points and the cross attention run on lrn_train_attention_* with the reference's dropout rate on the
        attention weights (src/model.py:84, nn.MultiheadAttention(dropout=0.1)); the query-side linears (self-attention
        projections, FFN, pos_emb layer 2, cross-attention q / out_proj) take the same bf16 tensor-core linear when the
        batch has >= 256 query rows; residual + LayerNorm is lrn_add_layernorm; point_mlp, dropouts and heads are stock
        ops.  Same parameters as DetrTransformerDecoderLayer; dropout draws differ from the reference's RNG stream (they
        would from run to run there, too)."""
        from .train_ops import (KVGradShare, add_layernorm, cross_attention_train, kv_proj, linear_bf16, pos_hidden_train,
                                self_attention_train, thin_linear)
        B, N, _ = context.shape
        d, H = self.d_model, 8
        wk = torch.cat([l.cross_attn.in_proj_weight[d:2 * d] for l in self.decoder_layers])
        wv = torch.cat([l.cross_attn.in_proj_weight[2 * d:] for l in self.decoder_layers])
        bk = torch.cat([l.cross_attn.in_proj_bias[d:2 * d] for l in self.decoder_layers])
        bv = torch.cat([l.cross_attn.in_proj_bias[2 * d:] for l in self.decoder_layers])
        mem = linear_bf16(fused_pm, self.context_proj.weight, self.context_proj.bias)      # (B,N,256) bf16
        h = pos_hidden_train(context, self.pos_emb.mlp[0].weight, self.pos_emb.mlp[0].bias)    # (B,N,256) bf16
        posm = linear_bf16(h, self.pos_emb.mlp[2].weight, self.pos_emb.mlp[2].bias)
        share = KVGradShare()                           # the attention backward writes dK / dV of all layers in place
        k_l = kv_proj(mem + posm, wk, bk, 6, H, share, key=True)  # six (B, H, N, 32) views of one (B, N, 6, H, 32) GEMM result
        v_l = kv_proj(mem, wv, bv, 6, H, share, key=False)
        rows = B * noisy_line.shape[1]
        tc = rows >= 256 and rows % 64 == 0   # query-side linears on the bf16 tensor-core path (fwd, dgrad, wgrad)
        lin16 = linear_bf16 if tc else F.linear   # self attention's [q | k] and v stay bf16 where the tensor-core linear produced them

        def lin(x, w, b):
            return linear_bf16(x, w, b, torch.float32) if tc else F.linear(x, w, b)

        pe0, pe2 = self.pos_emb.mlp[0], self.pos_emb.mlp[2]
        tgt = self.point_mlp(noisy_line.transpose(2, 1)).transpose(2, 1)
        current = noisy_line
        outs = []
        for i, (layer, head) in enumerate(zip(self.decoder_layers, self.reg_branches)):
            qpos = lin(F.relu(thin_linear(current, pe0.weight, pe0.bias)), pe2.weight, pe2.bias)
            sa = layer.self_attn
            att = self_attention_train(lin16(tgt + qpos, sa.in_proj_weight[:2 * d], sa.in_proj_bias[:2 * d]),
                                       lin16(tgt, sa.in_proj_weight[2 * d:], sa.in_proj_bias[2 * d:]), sa.dropout)
            att = lin(att, sa.out_proj.weight, sa.out_proj.bias)
            tgt = add_layernorm(tgt, layer.dropout1(att), layer.norm1)
            ca = layer.cross_attn
            qh = lin(tgt + qpos, ca.in_proj_weight[:d], ca.in_proj_bias[:d])
            att = cross_attention_train(qh, k_l[i], v_l[i], ca.dropout, share, i)
            tgt = add_layernorm(tgt, layer.dropout2(lin(att, ca.out_proj.weight, ca.out_proj.bias)), layer.norm2)
            ffn = lin(layer.dropout(F.relu(lin(tgt, layer.linear1.weight, layer.linear1.bias))), layer.linear2.weight, layer.linear2.bias)
            tgt = add_layernorm(tgt, layer.dropout3(ffn), layer.norm3)
            current = current + thin_linear(F.relu(lin(tgt, head[0].weight, head[0].bias)), head[2].weight, head[2].bias)   # reg_branches[i]: 256 -> 128 on the tensor cores
            outs.append(current - noisy_line)
        return torch.stack(outs)

    def forward(self, context, noisy_line):
        _require_cuda(context, "LineRefineNet")
        if context.dim() != 3 or noisy_line.dim() != 3 or context.shape[0] != noisy_line.shape[0] or context.shape[-1] != 4 \
                or noisy_line.shape[-1] != 3:
            raise ValueError(f"expected context (B,N,4) and noisy_line (B,M,3), got {tuple(context.shape)} and {tuple(noisy_line.shape)}")
        if not _use_native(self, context, noisy_line):
            enc = self.context_encoder
            if self.training and noisy_line.shape[1] == 32 and train_ops.native_train_supported(enc):
                _, fused_pm = train_ops.encoder_train_forward(enc, context, point_major=True)
                return self._refine_fast_train(context, noisy_line, fused_pm)
            _, fused = enc(context.transpose(2, 1))   # with native training on (M != 32): the channel-major native encoder
            memory = self.context_proj(fused.transpose(2, 1))
            return self._refine(context, noisy_line, memory, native_heads=False)
        B, N = context.shape[:2]
        # bf16 / tf32 tiers with M = 32: the native decoder; the fp32x3 tier and M != 32 keep the whole decoder in fp32
        # (stock attention / linears, native point_mlp and heads)
        native = self.precision != "fp32x3" and noisy_line.shape[1] == 32
        bf16 = native and self.precision == "bf16"
        if bf16:
            # ~1.2M context points per pass, up to 2048 segments: the query-side GEMMs (32 rows per segment) need
            # thousands of rows to fill the 74 CTA pairs, and no (B,N,1536) K / V temporaries exist on this path
            chunk = max(1, min(8 * self.segment_chunk, (4 * ops.DEFAULT_CHUNK_ROWS) // max(N, 1)))   # four full encoder waves
        elif native:
            chunk = max(1, min(self.segment_chunk, (1 << 20) // max(N, 1)))
        else:
            chunk = self.segment_chunk
        result = torch.empty(self.num_decoder_layers, *noisy_line.shape, dtype=torch.float32, device=context.device)
        for s in range(0, B, chunk):
            ctx = context[s:s + chunk].contiguous()
            line = noisy_line[s:s + chunk].contiguous()
            memory = self.context_encoder.run_native(ctx, pool=False, memory=True, memory_bf16=bf16)["memory"]
            if native:
                self._refine_native(ctx, line, memory, result[:, s:s + chunk])
            else:
                result[:, s:s + chunk] = self._refine(ctx, line, memory, native_heads=True)
        return result
