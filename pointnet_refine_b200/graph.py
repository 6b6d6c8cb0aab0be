"""CUDA-graph replay of the whole eval forward for a fixed (B, N): the reference's whole-scene loop runs the
model once per lane line with B = 1 (inference_whole_scene.py:130-139), where ~100 small launches, not the GPU,
set the latency.  Capture happens once; every call copies the inputs into static buffers and replays.

The captured launches hold raw pointers: the encoder's scratch buffer and every prepared weight (the BN-folded operand
blob, the folded decoder weights, the TF32-rounded copies).  The wrapper keeps all of them alive (warm-up and capture run
on the same side stream, so the scratch buffer the warm-up sized is the one the graph uses), and a replay after a
parameter change would silently use the old weights: call `recapture()` after load_state_dict / an optimizer step."""
from __future__ import annotations

import torch


class GraphedLineRefineNet:
    def __init__(self, model, B: int, N: int, M: int = 32):
        if model.training:
            raise RuntimeError("CUDA-graph replay is for eval-mode inference")
        dev = next(model.parameters()).device
        self.model = model
        self.ctx = torch.zeros(B, N, 4, dtype=torch.float32, device=dev)
        self.line = torch.zeros(B, M, 3, dtype=torch.float32, device=dev)
        self._side = torch.cuda.Stream(device=dev)
        self.recapture()

    def recapture(self):
        from . import ops
        model, dev = self.model, self.ctx.device
        side = self._side
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.no_grad(), torch.cuda.stream(side):      # warm-up: folds weights, sizes workspaces, sets kernel attributes
            for _ in range(3):
                model(self.ctx, self.line)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=side):
            self.out = model(self.ctx, self.line)
        # everything the captured kernels point at that the graph's own memory pool does not own; a copy of the prepared
        # weights, so that invalidate() or a rebuild by a later eager call cannot free what the graph reads
        self._keep = (ops.workspaces_of(dev), dict(model._prepared))

    @torch.no_grad()
    def __call__(self, context: torch.Tensor, noisy_line: torch.Tensor) -> torch.Tensor:
        self.ctx.copy_(context, non_blocking=True)
        self.line.copy_(noisy_line, non_blocking=True)
        self.graph.replay()
        return self.out


class GraphedTrainStep:
    """One training step of the reference's loop (train.py:56-72 / train_dist.py:168-189: zero_grad -> forward -> deep
    supervision loss -> backward -> optimizer.step()) captured ONCE as a CUDA graph and replayed per batch.

    Why: at 1024 x 1024 points the step is ~800 kernel launches; enqueuing them from Python takes ~58 ms of host time
    against ~63 ms of device time, so the step is host-bound as soon as the kernels get faster or several ranks share the
    host's cores (8 ranks: 82 ms per step eager).  A replay costs the host one call.

    What capture needs, and how the pieces provide it:
    * static shapes: `context` (B, N, 4), `noisy_line` (B, M, 3), `target` (B, M, 3) are copied into static buffers;
    * the optimizer's step count on the device: `FlatAdam` keeps it there (lrn_adam_step_capturable);
    * dropout that changes from replay to replay with frozen launch arguments: the train attention kernels add a device
      word to their seed (train_ops.DropoutSeedState), advanced inside the graph; torch's own dropout kernels take their
      Philox offsets from the graph-registered generator;
    * no host synchronisation anywhere in the step (there is none: the loss stays on the device).
    A frozen context encoder (`context_encoder.eval().requires_grad_(False)` with the native-training opt-in, FlatAdam over
    the trainable parameters only) runs as its eval forward inside the graph; the wrapper keeps the fold blob and scratch
    buffer that forward reads alive.
    Launch arguments are frozen at capture: the optimizer's lr / betas / eps / weight decay, the dropout rates and the batch
    shape are the ones in force when the step was built (the reference trains at a constant lr, train.py:21,40); build a
    new GraphedTrainStep to change them.
    `net` may be the bare model or `FlatDataParallel(model)`: its buffer broadcast and the flat-gradient all-reduce are
    NCCL launches on the capture stream and become graph nodes.  Parameters, Adam moments, BatchNorm buffers and the
    step count are snapshotted before the eager warm-up steps and restored after them, so construction does not train.

    If eager steps ran before construction, drop what they returned first (`del loss`): a live autograd graph keeps its
    AccumulateGrad nodes bound to the stream those steps ran on, and the capture then fails with
    cudaErrorStreamCaptureImplicit.

    __call__ returns (loss, pred_stack): static tensors, overwritten by the next call.  A batch of another shape (the ragged
    last batch of an epoch) runs the same step eagerly (`eager`)."""

    def __init__(self, net, optimizer, context, noisy_line, target, loss_fn=None, warmup: int = 2):
        from . import ops, train_ops
        from .optim import FlatAdam, deep_supervision_l1
        if not isinstance(optimizer, FlatAdam):
            raise TypeError("GraphedTrainStep needs FlatAdam: the step count must live on the device")
        model = getattr(net, "module", net)
        if not model.training:
            raise RuntimeError("GraphedTrainStep captures a training step: call model.train() first")
        dev = context.device
        self.net, self.model, self.opt = net, model, optimizer
        self.loss_fn = loss_fn or deep_supervision_l1
        self.ctx, self.line, self.tgt = (t.detach().clone().contiguous() for t in (context, noisy_line, target))
        self._seed = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).to(dev)      # host generator: follows torch.manual_seed
        self._params = [p for p, _ in optimizer._views]
        self._side = torch.cuda.Stream(device=dev)
        # ---- eager warm-up on the capture stream (lazy handles, kernel attributes, allocator), state put back afterwards
        keep = [optimizer._flat, optimizer._m, optimizer._v, optimizer._step_dev] + [b for b in model.buffers()]
        saved = [t.clone() for t in keep]
        self._side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self._side):
            for _ in range(warmup):
                self._step_body()
            with torch.no_grad():
                for t, s in zip(keep, saved):
                    if not torch.equal(t, s):   # what the step left alone (a frozen encoder's BatchNorm statistics) keeps
                        t.copy_(s)              # its version, so its prepared weights (encoder fold) are not rebuilt in the capture
        torch.cuda.current_stream(dev).wait_stream(self._side)
        # ---- capture
        self.graph = torch.cuda.CUDAGraph()
        train_ops.DropoutSeedState.word, train_ops.DropoutSeedState.calls = self._seed, 0
        try:
            with torch.cuda.graph(self.graph, stream=self._side):
                self._seed.add_(0x2545F4914F6CDD1D)        # every replay: a new dropout stream for the attention kernels
                loss, pred = self._step_body()
        except RuntimeError as e:
            if "capturing" in str(e) or "capture" in str(e):
                raise RuntimeError(
                    "GraphedTrainStep: the CUDA-graph capture of the train step failed.  The usual cause is an autograd graph "
                    "kept alive from an earlier eager step (e.g. a `loss` tensor still referenced): its AccumulateGrad nodes "
                    "stay bound to the stream that step ran on.  Drop those references (`del loss`) or keep only "
                    "`loss.detach()` / `loss.item()`, then build the step again.") from e
            raise
        finally:
            train_ops.DropoutSeedState.word = None
        self.loss, self.pred = loss.detach(), pred.detach()
        # what the captured kernels point at outside the graph's memory pool (a frozen encoder's eval forward: its fold blob
        # and scratch buffer), kept alive whatever later eager calls or invalidate() do to the caches
        self._keep = (ops.workspaces_of(dev), dict(model._prepared))
        self.replays = 0

    def close(self):
        """Destroy the captured graph and its memory pool.  Call it before torch.distributed.destroy_process_group() when
        the step ran under FlatDataParallel: NCCL's communicator teardown waits for every CUDA graph that holds one of its
        collectives."""
        import gc
        dev = self.ctx.device
        torch.cuda.synchronize(dev)
        self.graph = self.loss = self.pred = None
        gc.collect()
        torch.cuda.synchronize(dev)

    def _step_body(self):
        self.opt.zero_grad()
        pred = self.net(self.ctx, self.line)
        loss = self.loss_fn(pred, self.tgt)
        loss.backward()
        self.opt.step()
        return loss, pred

    def eager(self, context, noisy_line, target):
        """The same step launched kernel by kernel, for a batch whose shape differs from the captured one (the ragged last
        batch of an epoch when the DataLoader does not drop it).  Shares the optimizer state, the device step count and the
        parameters with the replays; returns (loss, pred_stack) detached."""
        self.opt.zero_grad()
        pred = self.net(context, noisy_line)
        loss = self.loss_fn(pred, target)
        loss.backward()
        self.opt.step()
        return loss.detach(), pred.detach()

    def __call__(self, context, noisy_line, target):
        if context.shape != self.ctx.shape or noisy_line.shape != self.line.shape or target.shape != self.tgt.shape:
            return self.eager(context, noisy_line, target)
        self.ctx.copy_(context, non_blocking=True)
        self.line.copy_(noisy_line, non_blocking=True)
        self.tgt.copy_(target, non_blocking=True)
        self.graph.replay()
        self.replays += 1
        # the replayed kernels wrote the parameters through raw pointers: the weight-folding caches of the eval path
        # fingerprint (data_ptr, _version)
        torch.autograd.graph.increment_version(self._params)
        return self.loss, self.pred
