"""EWC importance and penalty (SURVEY.md 8f-4) - drop-in for the EWC part of
``BRNullSpaceRunner`` (mmdet/engine/runner/nsrunner_roi_replay.py).

Mirrored surface:

* ``register_params(model)``            - :1006-1031 (names containing "bn", not "teacher_model")
* ``EWCImportance``                     - the accumulation loop body and tail of
  ``calculate_save_importance`` (:946-990): ``accumulate()`` after every backward,
  ``finish()`` appends to ``ewc_reg_terms`` and ``save()`` pickles
  ``ewc_reg_terms_ewc.pth`` in the reference's format
* ``EWCHook(module, reg_params, ewc_reg_terms)`` - :1038-1073, wraps ``module.loss`` and adds
  ``ewc_loss`` = 1000 * sum importance * (p - old)^2

What changed underneath: the reference runs ~8 tiny kernels per BatchNorm tensor per step
(two ``cat``, ``expand``, ``sub``, ``pow``, ``mul``, ``sum``, ``add`` - about a thousand
launches for R50-FPN's 106 BN tensors); here the penalty, its gradient and the importance
update are ONE multi-tensor launch each through the C ABI.
"""
from __future__ import annotations

import ctypes
import os.path as osp
from collections import defaultdict

import torch

from . import _lib
from ._lib import lib, check, EwcTensor


def register_params(model, must_names=("bn",), ignore_names=("teacher_model",)) -> dict:
    """:1006-1031 - ``{name: parameter}`` of the tensors EWC regularises: names that contain
    one of ``must_names`` (every name when that tuple is empty) and none of ``ignore_names``."""
    def wanted(name):
        if any(tag in name for tag in ignore_names):
            return False
        return not must_names or any(tag in name for tag in must_names)

    return {name: param for name, param in model.named_parameters() if wanted(name)}


def _table(n: int, device, cache: dict) -> torch.Tensor:
    # deterministic mode: the table also holds the penalty's fp64 partial sums
    det = _lib.deterministic()
    need = int(lib.nsgp_ewc_table_bytes(n))
    t = cache.get("table")
    if t is None or t.numel() < need or t.device != device or cache.get("det") != det:
        t = torch.empty(need, dtype=torch.uint8, device=device)
        cache["table"], cache["det"] = t, det
    return t


class EWCImportance:
    """Diagonal Fisher accumulation of ``calculate_save_importance`` (:946-990)."""

    def __init__(self, reg_params: dict):
        self.reg_params = reg_params
        self.importance = {n: p.clone().detach().fill_(0) for n, p in reg_params.items()}   # :955-956
        self._cache = {}

    @torch.no_grad()
    def accumulate(self, len_data_batch: int, len_dataloader: int):
        """``importance[n] += grad**2 * len(data_batch) / len(dataloader)`` for every
        registered parameter with a gradient (:978-981) - one launch."""
        items = [(self.importance[n], p.grad) for n, p in self.reg_params.items()
                 if p.grad is not None]
        if not items:
            return
        dev = items[0][0].device
        arr = (EwcTensor * len(items))()
        keep = []
        for k, (imp, g) in enumerate(items):
            _lib.require_cuda(imp, "importance")
            if g.dtype != torch.float32 or not g.is_contiguous():
                g = g.float().contiguous()
            keep.append(g)
            arr[k].p, arr[k].importance = g.data_ptr(), imp.data_ptr()
            arr[k].numel, arr[k].tasks = imp.numel(), 0
        table = _table(len(items), dev, self._cache)
        check(lib.nsgp_ewc_accumulate(arr, len(items), float(len_data_batch),
                                      float(len_dataloader), table.data_ptr(), table.numel(),
                                      _lib.current_stream(dev)), "nsgp_ewc_accumulate")

    def all_reduce(self, group=None, average=True):
        """Not in the reference: there every rank keeps the importance of its own data shard
        (``calculate_save_importance`` never reduces over ranks, SURVEY 8f-4) and rank 0's file
        wins.  Call this before ``finish`` to use the whole dataset: mean (default) or sum of
        the per-rank importances, one all-reduce per tensor issued together."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        works = [dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=True)
                 for t in self.importance.values()]
        for w in works:
            w.wait()
        if average:
            world = dist.get_world_size(group)
            for t in self.importance.values():
                t.div_(world)

    def finish(self, ewc_reg_terms: dict = None) -> dict:
        """:951-953, 985-987 - append this task's importance and parameters."""
        if not ewc_reg_terms:
            ewc_reg_terms = {"importance": defaultdict(list), "task_param": defaultdict(list)}
        for n, p in self.reg_params.items():
            ewc_reg_terms["importance"][n].append(self.importance[n].unsqueeze(0))
            ewc_reg_terms["task_param"][n].append(p.unsqueeze(0).clone().detach())
        return ewc_reg_terms

    @staticmethod
    def save(ewc_reg_terms: dict, work_dir: str):
        torch.save(ewc_reg_terms, osp.join(work_dir, "ewc_reg_terms_ewc.pth"))        # :989


def load_importance(previous_dir: str, device) -> dict:
    """:996-999."""
    return torch.load(osp.join(previous_dir, "ewc_reg_terms_ewc.pth"), map_location=device)


class _EwcPenalty(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hook, *params):
        dev = params[0].device
        n = len(params)
        arr = hook._tensor_table(params)
        table = _table(n, dev, hook._cache)
        loss = torch.empty(1, dtype=torch.float64, device=dev)
        check(lib.nsgp_ewc_penalty(arr, n, float(hook.coeff), loss.data_ptr(), table.data_ptr(),
                                   table.numel(), _lib.current_stream(dev)), "nsgp_ewc_penalty")
        ctx.hook = hook
        ctx.save_for_backward(*params)
        return loss.to(torch.float32).reshape(())

    @staticmethod
    def backward(ctx, gout):
        hook = ctx.hook
        params = ctx.saved_tensors
        dev = params[0].device
        n = len(params)
        # one zero-filled allocation for all gradients, handed back as views
        sizes = [p.numel() for p in params]
        flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        arr = hook._tensor_table(params)
        base, off = flat.data_ptr(), 0
        for k in range(n):
            arr[k].grad = base + 4 * off
            off += sizes[k]
        go = gout.detach().to(torch.float32).reshape(1).contiguous()
        table = _table(n, dev, hook._cache)
        check(lib.nsgp_ewc_penalty_backward(arr, n, float(hook.coeff), go.data_ptr(),
                                            table.data_ptr(), table.numel(),
                                            _lib.current_stream(dev)),
              "nsgp_ewc_penalty_backward")
        grads = [g.view(p.shape) for g, p in zip(flat.split(sizes), params)]
        return (None,) + tuple(grads)


class EWCHook:
    """Same constructor and call contract as the reference class (:1038-1073):
    ``model.loss = EWCHook(module=model, reg_params=..., ewc_reg_terms=...)`` (:565).

    ``check_nonzero`` keeps the reference's ``if reg_loss["ewc_loss"] != 0`` (:1070), which
    costs one host sync per step; ``False`` always reports the key."""

    coeff = 1000.0

    def __init__(self, module, reg_params, ewc_reg_terms, check_nonzero=True):
        self.module = module
        self.reg_params = reg_params
        self.ewc_reg_terms = ewc_reg_terms
        self.ori_loss = module.loss
        self.check_nonzero = check_nonzero
        self._cache = {}
        self._stacks = None
        self._stack_key = None

    def _prepare(self):
        names = [n for n, p in self.reg_params.items() if p.requires_grad]          # :1060-1061
        key = tuple((n, len(self.ewc_reg_terms["importance"][n])) for n in names)
        if key != self._stack_key:
            stacks = []
            for n in names:
                p = self.reg_params[n]
                _lib.require_cuda(p, "parameter " + n)
                imp = torch.cat(self.ewc_reg_terms["importance"][n], dim=0)         # :1062-1063
                old = torch.cat(self.ewc_reg_terms["task_param"][n], dim=0)         # :1064-1065
                imp = imp.to(device=p.device, dtype=torch.float32).contiguous()
                old = old.to(device=p.device, dtype=torch.float32).contiguous()
                stacks.append((imp, old, imp.shape[0]))
            self._stacks, self._stack_key = stacks, key
        return [self.reg_params[n] for n in names]

    def _tensor_table(self, params):
        """Host table of the registered tensors; rebuilt only when an address changes."""
        # parameter addresses AND the stacks they are paired with: a rebuilt stack (a task was
        # appended to ewc_reg_terms) has new storage even when no parameter moved
        key = (tuple(p.data_ptr() for p in params), self._stack_key,
               tuple((imp.data_ptr(), old.data_ptr()) for imp, old, _ in self._stacks))
        if self._cache.get("arr_key") != key:
            arr = (EwcTensor * len(params))()
            for k, (p, (imp, old, tasks)) in enumerate(zip(params, self._stacks)):
                arr[k].p, arr[k].importance, arr[k].old_params = p.data_ptr(), imp.data_ptr(), old.data_ptr()
                arr[k].numel, arr[k].tasks = p.numel(), tasks
            self._cache["arr"], self._cache["arr_key"] = arr, key
        return self._cache["arr"]

    def penalty(self):
        params = self._prepare()
        if not params:
            return 0
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise _lib.NsgpError("EWC parameters must be contiguous fp32 tensors")
        return _EwcPenalty.apply(self, *params)

    def __call__(self, *args, **kwargs):
        result = self.ori_loss(*args, **kwargs)
        ewc = self.penalty()
        if isinstance(ewc, torch.Tensor) and (not self.check_nonzero or bool(ewc != 0)):   # :1070
            result.update({"ewc_loss": ewc})
        return result
