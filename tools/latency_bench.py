"""Single-line latency (the reference's whole-scene loop calls the model with B = 1, N = 1024 per lane line,
inference_whole_scene.py:130-139): eager launches vs one CUDA-graph replay."""
import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pointnet_refine_b200 as prb
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1
N = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
dev = torch.device("cuda:0")
m = prb.LineRefineNet().to(dev).eval()
ctx = torch.randn(B, N, 4, device=dev); line = torch.randn(B, 32, 3, device=dev)
def timeit(f, n=50):
    for _ in range(5): f()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e3
with torch.no_grad():
    eager = timeit(lambda: m(ctx, line))
    ref = m(ctx, line).clone()
    runner = prb.GraphedLineRefineNet(m, B, N)
    graphed = timeit(lambda: runner(ctx, line))
    out = runner(ctx, line)
print(json.dumps({"B": B, "N": N, "eager_ms": round(eager, 3), "cuda_graph_ms": round(graphed, 3),
                  "graph_vs_eager_max_abs": float((out - ref).abs().max())}))
