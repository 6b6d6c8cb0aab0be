"""Data-parallel training step (reference train_dist.py:143-189) on the native train path: one process per GPU, NCCL.
Runs the same step under (a) torch's DistributedDataParallel, exactly as train_dist.py:147 wraps the model, and (b)
pointnet_refine_b200.FlatDataParallel + FlatAdam (one flat gradient buffer, one all-reduce, one Adam
launch).  Checks for both that gradients are averaged and identical on all ranks and that parameters stay in sync,
that (a) and (b) produce the same averaged gradients, and prints the step times.  Launch with torchrun.
LRN_DDP_FROZEN=1 runs the transfer-learning step instead: context encoder frozen (`.eval().requires_grad_(False)`), both
optimizers over the trainable parameters only; frozen parameters get no gradient and no all-reduce, and with NCCL the
step is also captured as a GraphedTrainStep with FlatDataParallel's all-reduce inside the graph."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from torch.nn.parallel import DistributedDataParallel as DDP
import pointnet_refine_b200 as prb
from pointnet_refine_b200 import optim as lrn_optim

rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
backend = os.environ.get("LRN_DDP_BACKEND", "nccl")
frozen = os.environ.get("LRN_DDP_FROZEN") == "1"
if os.environ.get("LRN_DDP_ONE_GPU") == "1":      # single-GPU box: every rank on cuda:0, gloo as the transport (NCCL refuses
    local = 0                                     # two ranks on one device); exercises the same hooks / flat buffers / kernels
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if backend == "nccl":
    dist.init_process_group("nccl", device_id=dev)
else:
    dist.init_process_group(backend)


def barrier():
    if backend == "nccl":
        dist.barrier(device_ids=[local])
    else:
        dist.barrier()
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
N = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
g = torch.Generator(device=dev).manual_seed(100 + rank)                    # different shard per rank
ctx = torch.randn(B, N, 4, device=dev, generator=g)
line = torch.randn(B, 32, 3, device=dev, generator=g)
tgt = 0.1 * torch.randn(B, 32, 3, device=dev, generator=g)


def same_on_all_ranks(t):
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return float((hi - lo).abs().max())


def make_model():
    torch.manual_seed(0)
    model = prb.LineRefineNet().to(dev).train()
    model.context_encoder.native_training = True            # opt-in: sm_100a train path
    if frozen:
        model.context_encoder.eval().requires_grad_(False)
    for mod in model.modules():                              # dropout off: (a) and (b) must see the same function
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0
    return model, [p for p in model.parameters() if p.requires_grad]


def run(kind):
    model, trainable = make_model()
    if kind == "ddp":
        net = DDP(model, device_ids=[local], find_unused_parameters=True)      # as train_dist.py:147
        opt = torch.optim.Adam(trainable, lr=1e-3)
    else:
        net = prb.FlatDataParallel(model)
        opt = lrn_optim.FlatAdam(trainable, lr=1e-3)
        assert opt._grad is net.flat.grad, "FlatAdam must adopt FlatDataParallel's flat buffers"
    times, grads = [], None
    for it in range(5):
        torch.cuda.synchronize(); barrier(); t0 = time.perf_counter()
        opt.zero_grad()
        out = net(ctx, line)
        loss = lrn_optim.deep_supervision_l1(out, tgt)
        loss.backward()
        if it == 0:
            worst = 0.0
            for n, p in model.named_parameters():
                if not p.requires_grad:
                    assert p.grad is None, n
                    continue
                assert p.grad is not None, n
                worst = max(worst, same_on_all_ranks(p.grad))
            assert worst == 0.0, f"{kind}: gradients differ across ranks after the all-reduce: {worst}"
            grads = torch.cat([p.grad.detach().reshape(-1).clone() for p in trainable])
        opt.step()
        torch.cuda.synchronize(); times.append(time.perf_counter() - t0)
    chk = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum()
    assert same_on_all_ranks(chk) == 0.0, f"{kind}: parameters diverged across ranks"
    return grads, min(times[1:]), float(loss.detach()), getattr(net, "allreduce_calls", None)


g_ddp, t_ddp, loss_ddp, _ = run("ddp")
g_flat, t_flat, loss_flat, calls = run("flat")
rel = float((g_flat - g_ddp).norm() / g_ddp.norm())
# same function; run-to-run the fp32 atomics (batch statistics, split-K) sum in a different order and a few bf16 roundings
# flip, which is the same noise the gradient parity test allows (tests/test_gpu_train.py: 2e-2)
assert rel <= 2e-2, f"flat-buffer gradients differ from DDP's: rel-L2 {rel}"
graphed = None
if frozen and backend == "nccl":      # gloo collectives cannot be captured in a CUDA graph
    model, trainable = make_model()
    net = prb.FlatDataParallel(model)
    opt = lrn_optim.FlatAdam(trainable, lr=1e-3, capturable=True)
    step = prb.GraphedTrainStep(net, opt, ctx, line, tgt)
    graphed = [float(step(ctx, line, tgt)[0]) for _ in range(5)]
    chk = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum()
    assert same_on_all_ranks(chk) == 0.0, "graphed frozen step: parameters diverged across ranks"
    assert all(l == l and abs(l) < float("inf") for l in graphed), graphed
    step.close()
if rank == 0:
    print("ddp ok: " + json.dumps({"world": world, "backend": backend, "segments_per_rank": B, "points": N, "loss_ddp": round(loss_ddp, 5),
                                   "loss_flat": round(loss_flat, 5), "grad_rel_l2_flat_vs_ddp": rel,
                                   "step_ms_ddp_adam": round(1e3 * t_ddp, 2), "step_ms_flat_dp_flat_adam": round(1e3 * t_flat, 2),
                                   "segments_per_s_flat": round(world * B / t_flat), "allreduce_calls_per_step": calls // 5,
                                   "frozen_encoder": frozen, "graphed_losses": graphed}))
dist.destroy_process_group()
