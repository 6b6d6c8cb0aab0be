"""Training-loop machinery on the native kernels (SURVEY.md section 8f row 4).

`FlatAdam` is a drop-in for `optim.Adam(model.parameters(), lr=LR)` (reference train.py:40, train_dist.py:149): every
parameter becomes a view of ONE flat fp32 buffer (and its `.grad` a view of one flat gradient buffer), so a step is one
`lrn_adam_step_capturable` call instead of a multi-tensor sweep, and `zero_grad` is one memset.
`deep_supervision_l1` is the loss of train.py:63-69 (mean over decoder layers of L1Loss) as one fused forward+backward
kernel."""
from __future__ import annotations

import torch

from .flat import FlatParams
from .ops import _call


class FlatAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, capturable=False):
        params = [p for p in params]
        if not params:
            raise ValueError("FlatAdam got an empty parameter list")
        if any((not p.is_cuda) or p.dtype != torch.float32 for p in params):
            raise TypeError("FlatAdam expects CUDA float32 parameters (no CPU fallback)")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        if len(self.param_groups) != 1:
            raise ValueError("FlatAdam keeps ONE flat buffer: pass a plain parameter list, not several parameter groups")
        self._fp = FlatParams.of(params) or FlatParams(params)     # shared with ddp.FlatDataParallel when it wrapped the model first
        self._flat, self._grad = self._fp.flat, self._fp.grad
        self._m = torch.zeros_like(self._flat)
        self._v = torch.zeros_like(self._flat)
        self._views = list(zip(self._fp.params, self._fp.grad_views))
        # the step count lives on the device and the bias corrections are computed there, so step() can be captured in a
        # CUDA graph and replayed (graph.GraphedTrainStep).  `capturable` (torch.optim.Adam's flag of the same name) is
        # accepted for drop-in use and has no effect: every step is capturable.
        self._step_dev = torch.zeros(1, dtype=torch.int64, device=self._flat.device)

    @property
    def steps_taken(self) -> int:
        return int(self._step_dev.item())

    def _attach(self, keep_foreign: bool = True):
        """Make every parameter's .grad the view of the flat gradient buffer.  A gradient some other code bound to
        .grad meanwhile (e.g. DistributedDataParallel(gradient_as_bucket_view=True), set_to_none) is copied in when
        `keep_foreign` -- i.e. in step(), where it is THIS step's gradient -- and dropped in zero_grad()."""
        self._fp.attach(keep_foreign)

    def add_param_group(self, param_group):
        if getattr(self, "_views", None) is not None:
            raise ValueError("FlatAdam: parameter groups cannot be added after construction (one flat buffer)")
        super().add_param_group(param_group)

    def zero_grad(self, set_to_none: bool = False):
        self._attach(keep_foreign=False)     # rebind first: a stale foreign .grad must not be copied into the zeroed buffer
        self._grad.zero_()

    def state_dict(self):
        """Adam moments and the step count live in the flat buffers, not in `self.state`: add them to the checkpoint."""
        sd = super().state_dict()
        sd["flat_adam"] = {"exp_avg": self._m.clone(), "exp_avg_sq": self._v.clone(), "step": self.steps_taken}
        return sd

    def load_state_dict(self, state_dict):
        state_dict = dict(state_dict)
        flat = state_dict.pop("flat_adam", None)
        super().load_state_dict(state_dict)
        if flat is not None:
            if flat["exp_avg"].numel() != self._m.numel():
                raise ValueError("FlatAdam.load_state_dict: checkpoint belongs to a different parameter list")
            self._m.copy_(flat["exp_avg"])
            self._v.copy_(flat["exp_avg_sq"])
            self._step_dev.fill_(int(flat["step"]))

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self._attach()
        g = self.param_groups[0]
        hyper = (float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]))
        _call("lrn_adam_step_capturable", self._flat.device, self._flat, self._grad, self._m, self._v, self._flat.numel(),
              *hyper, self._step_dev)
        # the kernel wrote through raw pointers: tell autograd / the weight-folding caches (data_ptr + _version
        # fingerprints in model.py) that every parameter changed
        torch.autograd.graph.increment_version([p for p, _ in self._views])
        return loss


class _DeepSupervisionL1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target):
        L = pred.shape[0]
        pred_c, tgt_c = pred.detach().float().contiguous(), target.detach().float().contiguous()
        n = tgt_c.numel()
        if pred_c.numel() != L * n:
            raise ValueError(f"pred {tuple(pred.shape)} is not (L, *target.shape) for target {tuple(target.shape)}")
        loss = torch.empty((), dtype=torch.float32, device=pred.device)
        dpred = torch.empty_like(pred_c)
        _call("lrn_l1_deep_supervision", pred.device, pred_c, tgt_c, L, n, loss, dpred)
        ctx.save_for_backward(dpred)
        ctx.pred_dtype = pred.dtype
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (dpred,) = ctx.saved_tensors
        return (dpred * dloss).to(ctx.pred_dtype), None


def deep_supervision_l1(pred_stack: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """sum_l L1Loss(pred_stack[l], target) / L for pred_stack (L, B, M, 3), target (B, M, 3) (train.py:63-69)."""
    if not pred_stack.is_cuda:
        raise TypeError("deep_supervision_l1 expects CUDA tensors (no CPU fallback)")
    return _DeepSupervisionL1.apply(pred_stack, target)
