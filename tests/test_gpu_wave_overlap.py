"""bf16 encoder split into many back-to-back waves against the same input in one wave.

The chain and fusion kernels of consecutive waves overlap through programmatic dependent launch: a kernel starts while
the one before it is finishing and waits (griddepcontrol.wait) only before it touches the single operand buffer they
share (chain: write after the previous fusion's reads; fusion: read after its chain's writes; pooling atomics).  A
missing or misplaced wait shows up as operand rows of the wrong wave, i.e. max / argmax that differ from a run with no
wave boundary at all.  The max half of global_feat and the argmax do not depend on the order of the atomics, so they must
be bit-identical; the mean half is a sum of non-negative fp32 partials in another order."""
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu

WAVE = 74 * 256       # one 256-point tile per CTA pair of a 148-SM B200: every wave is short, a call is dozens of them
ONE_WAVE = 1 << 30    # chunk_rows beyond B * N: a single wave


@pytest.fixture(scope="module")
def enc():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import pointnet_refine_b200 as prb
    m = prb.LineRefineNet().to("cuda:0").eval()
    m.load_state_dict(synth.to_torch(synth.make_state_dict(0)), strict=True)
    m.precision = "bf16"
    return m.context_encoder


def _run(enc, ctx, chunk_rows, argmax):
    enc.chunk_rows = chunk_rows
    try:
        with torch.no_grad():
            return enc.run_native(ctx, pool=True, argmax=argmax)
    finally:
        enc.chunk_rows = 0


def _ctx(B, N, seed):
    return torch.randn(B, N, 4, device="cuda:0", generator=torch.Generator(device="cuda:0").manual_seed(seed))


def _assert_same(out, ref, N, argmax):
    gf, gr = out["global_feat"], ref["global_feat"]
    assert torch.isfinite(gf).all()
    assert torch.equal(gf[:, :1024], gr[:, :1024])
    if argmax:
        assert torch.equal(out["argmax"], ref["argmax"])
    # mean: at most N non-negative partials (each scaled by 1 / N) summed in another order; two orders of k non-negative
    # terms differ by at most 2 (k - 1) u times their sum
    bound = 2 * N * 2.0 ** -24 * gr[:, 1024:]
    assert ((gf[:, 1024:] - gr[:, 1024:]).abs() <= bound).all()


# N = 1000: segments straddle every wave and warps straddle segments (general pooling path); N = 2048 with pooling
# only: the fast path (every warp inside one segment)
@pytest.mark.parametrize("B,N,argmax", [(600, 1000, True), (300, 2048, False)])
def test_many_waves_match_one_wave(enc, B, N, argmax):
    ctx = _ctx(B, N, 7)
    assert B * N >= 30 * WAVE
    ref = _run(enc, ctx, ONE_WAVE, argmax)
    out = _run(enc, ctx, WAVE, argmax)
    _assert_same(out, ref, N, argmax)


def test_back_to_back_calls_of_different_batch(enc):
    """A second call with another B right behind the first one: its first chain kernel overwrites the operand buffer the
    first call's last fusion kernel reads."""
    c1, c2 = _ctx(500, 1000, 11), _ctx(237, 1000, 12)
    r1, r2 = _run(enc, c1, ONE_WAVE, True), _run(enc, c2, ONE_WAVE, True)
    torch.cuda.synchronize()
    o1 = _run(enc, c1, WAVE, True)
    o2 = _run(enc, c2, WAVE, True)
    _assert_same(o1, r1, 1000, True)
    _assert_same(o2, r2, 1000, True)


def test_graph_replay_matches_eager(enc):
    """A many-wave call captured in a CUDA graph (the programmatic launches become programmatic edges) and replayed."""
    B, N = 400, 1000
    ctx = _ctx(B, N, 13)
    eager = _run(enc, ctx, WAVE, True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):           # warm-up on the capture stream: its workspace and kernel attributes
        _run(enc, ctx, WAVE, True)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        captured = _run(enc, ctx, WAVE, True)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        _assert_same(captured, eager, N, True)
