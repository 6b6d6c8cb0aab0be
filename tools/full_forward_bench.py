"""Full LineRefineNet eval forward against the encoder alone: where does the time go?"""
import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pointnet_refine_b200 as prb
B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
N = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
dev = torch.device("cuda:0")
m = prb.LineRefineNet().to(dev).eval()
ctx = torch.randn(B, N, 4, device=dev); line = torch.randn(B, 32, 3, device=dev)
def timeit(f, n=3):
    for _ in range(2): f()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e3
with torch.no_grad():
    t_full = timeit(lambda: m(ctx, line))
    t_enc = timeit(lambda: m.context_encoder.run_native(ctx, pool=False, memory=True))
    t_pool = timeit(lambda: m.context_encoder.run_native(ctx, pool=True))
print(json.dumps({"B": B, "N": N, "full_forward_ms": round(t_full, 2), "encoder+proj_ms": round(t_enc, 2), "encoder_pool_ms": round(t_pool, 2),
                  "full_segments_per_s": round(B / t_full * 1e3, 1)}))
