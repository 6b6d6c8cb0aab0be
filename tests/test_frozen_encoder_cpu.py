"""CPU-only checks of LRN_OUT_FUSED_BF16, the encoder output that feeds the native train decoder from a frozen encoder:
the header declares it, the binding exports it, it adds no workspace to any flag set, and on its own it needs only the
operand rows (no point-major block for the projection)."""
import os
import re

from pointnet_refine_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAG_SETS = (_lib.OUT_POOL, _lib.OUT_ARGMAX, _lib.OUT_FUSED, _lib.OUT_MEMORY, _lib.OUT_POOL | _lib.OUT_ARGMAX,
             _lib.OUT_FUSED | _lib.OUT_MEMORY, _lib.OUT_POOL | _lib.OUT_ARGMAX | _lib.OUT_FUSED | _lib.OUT_MEMORY,
             _lib.OUT_MEMORY | _lib.OUT_MEMORY_BF16)


def test_header_declares_fused_bf16_flag():
    header = open(os.path.join(ROOT, "include", "lrn_b200.h")).read()
    m = re.search(r"^\s*LRN_OUT_FUSED_BF16\s*=\s*(\d+)\s*,", header, re.M)
    assert m and int(m.group(1)) == 32
    assert _lib.OUT_FUSED_BF16 == int(m.group(1))
    assert re.search(r"^#define LRN_ABI_VERSION 5$", header, re.M) and _lib.ABI_VERSION == 5   # additive: no version change


def test_fused_bf16_adds_no_workspace():
    ws = _lib.lib.lrn_encoder_workspace_bytes
    bf16 = _lib.PREC_BF16
    for B, N in ((1, 1), (1, 129), (3, 700), (7, 300), (74, 4096), (1024, 1024)):
        for chunk_rows in (0, 1, 128, 129, 512, 148 * 128 * 16):
            for flags in FLAG_SETS:
                assert ws(B, N, bf16, flags | _lib.OUT_FUSED_BF16, chunk_rows) == ws(B, N, bf16, flags, chunk_rows), \
                    (B, N, flags, chunk_rows)
            # alone: the operand rows of one wave, (chunk, 2048) bf16, and nothing for the projection
            chunk = min(-(-max(chunk_rows if chunk_rows > 0 else 148 * 128 * 16, 128) // 128) * 128, -(-B * N // 128) * 128)
            alone = ws(B, N, bf16, _lib.OUT_FUSED_BF16, chunk_rows)
            assert alone == -(-chunk * 2048 * 2 // 1024) * 1024, (B, N, chunk_rows)
            assert alone == ws(B, N, bf16, _lib.OUT_POOL, chunk_rows) < ws(B, N, bf16, _lib.OUT_MEMORY, chunk_rows)


def test_fused_bf16_refusals_need_no_device():
    """Flag combinations the library refuses before it looks for a device (LRN_ERR_BAD_ARG = 6), and no kernel is
    enqueued for them."""
    fwd = _lib.lib.lrn_encoder_forward
    fake = 1 << 20          # validation refuses before any pointer is dereferenced
    launches = _lib.launch_counter
    F = _lib.OUT_FUSED_BF16
    assert fwd(fake, _lib.PREC_BF16, fake, 2, 64, F | _lib.OUT_FUSED, None, fake, None, None, 0, fake, 1 << 30, None) == 6
    assert fwd(fake, _lib.PREC_TF32, fake, 2, 64, F, None, fake, None, None, 0, fake, 1 << 30, None) == 6
    assert fwd(fake, _lib.PREC_FP32X3, fake, 2, 64, F, None, fake, None, None, 0, fake, 1 << 30, None) == 6
    assert fwd(fake, _lib.PREC_BF16, fake, 2, 64, F, None, None, None, None, 0, fake, 1 << 30, None) == 6
    assert _lib.launch_counter == launches
