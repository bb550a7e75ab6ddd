"""
Optimizer / scheduler factory (reference: resnet/utils/optim_util.py:11-30).

`get_optimizer('SGD', model, args)` returns FusedSGD: a torch.optim.SGD subclass (same param_groups,
same state[p]['momentum_buffer'], same state_dict, works with lr schedulers and GradScaler) whose
step() is ONE multi-tensor kernel launch (b200_sgd_step) per parameter group instead of torch's
foreach kernels. 'Adam' and 'AdamW' likewise return FusedAdam / FusedAdamW (torch.optim.Adam / AdamW
subclasses, torch's state format, one b200_adam_step launch per parameter group). Any other optimizer
name resolves to torch.optim as in the reference.
"""
import importlib
from typing import Any, Dict, Optional

import torch

from pytorch_ddp_resnet_b200 import ops


def _same_layout(a: torch.Tensor, b: torch.Tensor) -> bool:
    """Same element order in memory (strides of size-1 dimensions do not matter)."""
    if a.shape != b.shape:
        return False
    return all(sa == sb for n, sa, sb in zip(a.shape, a.stride(), b.stride()) if n > 1)


class _FusedStepBase:
    """What every fused optimizer here shares: the pointer tables its one launch per group reads, and a
    device-resident learning rate per group. Mixed in before the torch.optim class it extends."""

    def _init_fused(self):
        self._tables = {}   # per (device, rows, n): ring of (pinned host table, device table, event)
        self._ring = 4
        self._lr_dev = {}   # (group index, device) -> [device fp32 scalar, value it holds]

    def _table(self, device, n, rows=4):
        """(pinned host table, device table, event) for this step's pointer upload. Eager steps rotate
        through a small ring (the host may run ahead of the copies); a CUDA-graph capture gets a
        dedicated pair that no later eager step overwrites, because every replay re-reads it."""
        key = (device, rows, n)
        ring = self._tables.get(key)
        if ring is None:
            def pair():
                return (torch.empty((rows, n), dtype=torch.int64).pin_memory(),
                        torch.empty((rows, n), dtype=torch.int64, device=device))
            ring = {"slot": 0, "bufs": [pair() + (torch.cuda.Event(),) for _ in range(self._ring)],
                    "used": [False] * self._ring, "capture": [], "pair": pair}
            self._tables[key] = ring
        if torch.cuda.is_current_stream_capturing():
            # every captured launch keeps its own table for the life of the graph (replays re-read it)
            if len(ring["capture"]) >= 256:
                raise RuntimeError(f"{type(self).__name__}: too many CUDA-graph captures of the same parameter set")
            ring["capture"].append(ring["pair"]())
            host, dev = ring["capture"][-1]
            return host, dev, None
        s = ring["slot"]
        ring["slot"] = (s + 1) % self._ring
        host, dev, ev = ring["bufs"][s]
        if ring["used"][s]:
            ev.synchronize()  # the copy issued `ring` steps ago has long finished
        ring["used"][s] = True
        return host, dev, ev

    def _upload(self, device, rows):
        """Fills a table with `rows` (lists of ints, one per table row) and starts its copy to the device."""
        n = len(rows[0])
        host, dev, ev = self._table(device, n, len(rows))
        for r, vals in enumerate(rows):
            host[r] = torch.tensor(vals, dtype=torch.int64)
        dev.copy_(host, non_blocking=True)
        if ev is not None:
            ev.record()
        return dev

    def _lr_tensor(self, gi, group, device):
        """Device-resident learning rate of a param group, refreshed whenever the scheduler moved it.
        The kernel reads it through a pointer, so a captured CUDA graph follows lr schedules."""
        key = (gi, device)
        slot = self._lr_dev.get(key)
        lr = float(group["lr"])
        if slot is None:
            slot = [torch.full((), lr, dtype=torch.float32, device=device), lr]
            self._lr_dev[key] = slot
        elif slot[1] != lr and not torch.cuda.is_current_stream_capturing():
            slot[0].fill_(lr)
            slot[1] = lr
        return slot[0]

    def sync_lr(self):
        """Pushes the current param_group lrs to their device scalars (call before a graph replay)."""
        for (gi, device) in list(self._lr_dev):
            self._lr_tensor(gi, self.param_groups[gi], device)

    def _amp_scaling(self):
        """(inv_scale, found_inf) device tensors a GradScaler handed over for this step, or (None, None)."""
        grad_scale = getattr(self, "grad_scale", None)
        found_inf = getattr(self, "found_inf", None)
        inv_scale = None
        if grad_scale is not None:
            inv_scale = grad_scale.double().reciprocal().float()
        return inv_scale, found_inf


class FusedSGD(_FusedStepBase, torch.optim.SGD):
    _step_supports_amp_scaling = True  # GradScaler hands us grad_scale / found_inf, no host sync

    def __init__(self, params, **kwargs):
        kwargs.pop("foreach", None)
        kwargs.pop("fused", None)
        super().__init__(params, **kwargs)
        self._init_fused()

    @torch.no_grad()
    def step_subset(self, params):
        """The update of `params` only (one launch): GraphedTrainStep steps every gradient bucket as soon as its
        exchange has finished, overlapped with the rest of backward, instead of all parameters at the end."""
        return self.step(only={id(p) for p in params})

    @torch.no_grad()
    def step(self, closure=None, only=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        inv_scale, found_inf = self._amp_scaling()
        for gi, group in enumerate(self.param_groups):
            if group.get("maximize", False):
                raise NotImplementedError("FusedSGD: maximize=True is not supported")
            fresh, seasoned = [], []
            for p in group["params"]:
                if p.grad is None or (only is not None and id(p) not in only):
                    continue
                if not p.is_cuda or p.dtype != torch.float32:
                    raise RuntimeError("FusedSGD needs fp32 CUDA parameters (no CPU fallback)")
                g = p.grad
                if g.is_sparse:
                    raise RuntimeError("FusedSGD does not support sparse gradients")
                if g.dtype != torch.float32 or not _same_layout(g, p):
                    g = torch.empty_like(p).copy_(g)
                state = self.state[p]
                buf0 = state.get("momentum_buffer")
                if buf0 is not None and not _same_layout(buf0, p):
                    # e.g. a reference checkpoint: NCHW-contiguous buffers for channels_last parameters;
                    # the kernel walks param / grad / buffer as flat memory, so they must share strides
                    state["momentum_buffer"] = torch.empty_like(p).copy_(buf0)
                if group["momentum"] != 0 and state.get("momentum_buffer") is None:
                    state["momentum_buffer"] = torch.empty_like(p)  # written by the kernel (buf = g)
                    fresh.append((p, g, state["momentum_buffer"]))
                else:
                    buf = state.get("momentum_buffer")
                    seasoned.append((p, g, buf if buf is not None else p))
            for items, first in ((fresh, True), (seasoned, False)):
                if not items:
                    continue
                n = len(items)
                device = items[0][0].device
                dev = self._upload(device, [[p.data_ptr() for p, _, _ in items], [g.data_ptr() for _, g, _ in items],
                                            [b.data_ptr() for _, _, b in items], [p.numel() for p, _, _ in items]])
                ops.sgd_step(dev, n, max(p.numel() for p, _, _ in items), group["lr"], group["momentum"],
                             group["dampening"], group["weight_decay"], group["nesterov"], first,
                             inv_scale=inv_scale, found_inf=found_inf,
                             lr_dev=self._lr_tensor(gi, group, device))
                for p, _, _ in items:
                    torch.autograd.graph.increment_version(p)
                self._keepalive = getattr(self, "_keepalive", [])[-64:] + [items]  # grads copied above outlive the launch
        return loss


class _FusedAdamBase(_FusedStepBase):
    """step() of torch.optim.Adam / AdamW as ONE b200_adam_step launch per parameter group.

    The state is torch's: state[p] holds `step` (a 0-d fp32 tensor on the parameter's device, the format of
    torch's fused and capturable Adam), `exp_avg`, `exp_avg_sq` and, with amsgrad, `max_exp_avg_sq`, the moments
    in the parameter's memory layout. The launch advances `step` on the device, so the update needs no host
    sync and a captured CUDA graph advances it at every replay; the learning rate is read from a device scalar
    (sync_lr), so lr schedulers keep working under a graph. state_dicts load from and into stock torch.optim
    Adam / AdamW, including a `step` saved as a Python int (torch 1.x) or a CPU tensor (torch 2.x)."""
    _step_supports_amp_scaling = True  # GradScaler hands us grad_scale / found_inf, no host sync

    def _check_kwargs(self, kwargs):
        kwargs.pop("foreach", None)
        kwargs.pop("fused", None)
        kwargs.pop("capturable", None)
        for flag in ("maximize", "differentiable"):
            if kwargs.get(flag, False):
                raise NotImplementedError(f"{type(self).__name__}: {flag}=True is not supported")
        return kwargs

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        # the device format right away (not lazily in step()): a CUDA-graph snapshot taken before the first step
        # must see the tensors the kernel will update
        for group in self.param_groups:
            for p in group["params"]:
                if self.state.get(p):
                    self._prepare_state(p, self.state[p])

    @staticmethod
    def _prepare_state(p, state):
        """step as a 0-d fp32 tensor on p's device; moments in p's memory layout (a state_dict saved from
        NCHW-contiguous parameters, or by torch on the host, is re-laid-out for channels_last filters)."""
        step = state.get("step")
        if step is not None and not (torch.is_tensor(step) and step.dtype == torch.float32 and step.dim() == 0
                                     and step.device == p.device):
            state["step"] = torch.as_tensor(step).detach().reshape(()).to(dtype=torch.float32, device=p.device,
                                                                          copy=True)
        for key in ("exp_avg", "exp_avg_sq", "max_exp_avg_sq"):
            buf = state.get(key)
            if buf is not None and not (buf.device == p.device and buf.dtype == p.dtype and _same_layout(buf, p)):
                state[key] = torch.empty_like(p).copy_(buf)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        inv_scale, found_inf = self._amp_scaling()
        name = type(self).__name__
        for gi, group in enumerate(self.param_groups):
            for flag in ("maximize", "differentiable"):
                if group.get(flag, False):
                    raise NotImplementedError(f"{name}: {flag}=True is not supported")
            amsgrad = bool(group["amsgrad"])
            items = []
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda or p.dtype != torch.float32:
                    raise RuntimeError(f"{name} needs fp32 CUDA parameters (no CPU fallback)")
                g = p.grad
                if g.is_sparse:
                    raise RuntimeError(f"{name} does not support sparse gradients")
                if g.dtype != torch.float32 or not _same_layout(g, p):
                    g = torch.empty_like(p).copy_(g)
                state = self.state[p]
                if len(state) == 0:
                    # fresh state (torch: step 0, zero moments); created eagerly, before any graph capture
                    state["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
                    state["exp_avg"] = torch.zeros_like(p)
                    state["exp_avg_sq"] = torch.zeros_like(p)
                if amsgrad and "max_exp_avg_sq" not in state:
                    state["max_exp_avg_sq"] = torch.zeros_like(p)
                items.append((p, g, state))
            if not items:
                continue
            device = items[0][0].device
            v = [st["exp_avg_sq"] for _, _, st in items]
            vmax = [st["max_exp_avg_sq"] for _, _, st in items] if amsgrad else v
            dev = self._upload(device, [[p.data_ptr() for p, _, _ in items], [g.data_ptr() for _, g, _ in items],
                                        [st["exp_avg"].data_ptr() for _, _, st in items], [t.data_ptr() for t in v],
                                        [t.data_ptr() for t in vmax], [st["step"].data_ptr() for _, _, st in items],
                                        [p.numel() for p, _, _ in items]])
            beta1, beta2 = group["betas"]
            ops.adam_step(dev, len(items), max(p.numel() for p, _, _ in items), group["lr"], beta1, beta2,
                          group["eps"], group["weight_decay"], group["decoupled_weight_decay"], amsgrad,
                          inv_scale=inv_scale, found_inf=found_inf, lr_dev=self._lr_tensor(gi, group, device))
            for p, _, _ in items:
                torch.autograd.graph.increment_version(p)
            self._keepalive = getattr(self, "_keepalive", [])[-64:] + [items]  # grads copied above outlive the launch
        return loss


class FusedAdam(_FusedAdamBase, torch.optim.Adam):
    """torch.optim.Adam (decoupled_weight_decay=True gives AdamW's update) with a fused sm_100a step()."""

    def __init__(self, params, **kwargs):
        super().__init__(params, **self._check_kwargs(kwargs))
        self._init_fused()


class FusedAdamW(_FusedAdamBase, torch.optim.AdamW):
    """torch.optim.AdamW (decoupled weight decay, default 0.01) with a fused sm_100a step()."""

    def __init__(self, params, **kwargs):
        super().__init__(params, **self._check_kwargs(kwargs))
        self._init_fused()


_FUSED = {"SGD": FusedSGD, "Adam": FusedAdam, "AdamW": FusedAdamW}


def get_optimizer(optimizer_cls_name: str, model, optimizer_args: Dict[str, Any]):
    if optimizer_cls_name in _FUSED:
        return _FUSED[optimizer_cls_name](model.parameters(), **optimizer_args)
    optimizer_cls = getattr(importlib.import_module("torch.optim"), optimizer_cls_name)
    return optimizer_cls(model.parameters(), **optimizer_args)


def get_scheduler(scheduler_cls_name: str, optimizer, scheduler_args: Dict[str, Any]) -> Optional[Any]:
    if scheduler_cls_name == "None":
        return None
    scheduler_cls = getattr(importlib.import_module("torch.optim.lr_scheduler"), scheduler_cls_name)
    return scheduler_cls(optimizer, **scheduler_args)
