"""``SGDNSCL`` - SGD with null-space gradient projection, drop-in for
mmdet/engine/optimizers/SGD_NSCL.py:15-415.

Same constructor, param-group keys (``names``, ``svd``), public state
(``eigens``, ``transforms``, ``state[p]['previous_grad'|'step']``) and methods
(``get_eigens``, ``get_transforms``, ``adaptive_threshold``, ``step``).

What changed underneath
* ``step``: ONE C-ABI call.  A fused multi-tensor kernel does the weight decay
  (in place on ``p.grad``, :399-400), the momentum buffer (:402-411) and
  ``-lr * buf`` for every parameter; protected layers then get
  ``W += update.view(Cout,-1) @ P`` (:82-95) from the 3xTF32 tensor-core
  contraction with the add fused in its epilogue.
* ``get_eigens``: symmetric eigendecomposition on the GPU (cuSOLVER syevd through
  ``torch.linalg.eigh``, fp64 by default) instead of a full fp32 SVD (:377);
  for a PSD matrix the singular values / right singular vectors are the
  eigenpairs sorted by descending magnitude.  Runs once per task boundary.
"""
from __future__ import annotations

import ctypes
from collections import defaultdict

import numpy as np
import scipy.ndimage
import torch
from torch.optim.optimizer import Optimizer

from . import _lib
from ._lib import lib, check, ptr, SgdTensor, ProjLayer, SgdPlan


class SGDNSCL(Optimizer):
    def __init__(self, params, lr=1e-3, momentum=0, dampening=0, nesterov=False, svd=False,
                 thres=1.001, weight_decay=0, eig_dtype=torch.float64):
        if not 0.0 <= lr:
            raise ValueError("Invalid learning rate: {}".format(lr))
        defaults = dict(lr=lr, momentum=momentum, dampening=dampening, nesterov=nesterov,
                        weight_decay=weight_decay, svd=svd, thres=thres)
        super().__init__(params, defaults)
        self.eigens = defaultdict(dict)
        self.transforms = defaultdict(dict)
        self.count = 0
        self.eig_dtype = eig_dtype
        self._prepared = {}     # name -> (key, pt_hi, pt_lo)
        self._stage = {}        # name -> (u_hi, u_lo)
        self._workspace = None
        self._plans = {}        # group index -> cached tables / T arena / plan (_build_group_cache)
        self._lowrank = {}      # name -> (P tensor, P._version, U (d,r), scale) from get_transforms
        self._lowrank_prepared = {}
        self.lowrank_max_ratio = 0.25   # use G - (G U) U^T while r <= ratio * d

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:
            group.setdefault("svd", False)
            group.setdefault("names", [])

    # ------------------------------------------------------------ projector build
    def adaptive_threshold(self, svals: torch.Tensor, offset: float = 0):
        """Boolean mask over the spectrum, True from the elbow index on
        (SGD_NSCL.py:98-177; host numpy/scipy exactly as there)."""
        pts = svals.detach().cpu().numpy()
        assert pts.ndim == 1
        n = len(pts)
        if n >= 128:
            sm = scipy.ndimage.gaussian_filter1d(pts, sigma=10)
            first = sm[:-1] - sm[1:]
            second = first[:-1] - first[1:]
            drop = int(n * 0.03 / 2)
            assert n - drop >= 10
            inner = second[drop:-drop]
            elbow_val = pts[np.argmax(inner) + int((n - len(inner)) / 2)]
        else:
            first = pts[:-1] - pts[1:]
            second = first[:-1] - first[1:]
            elbow_val = pts[np.argmax(second) + int((n - len(second)) / 2)]
        i_thres = np.arange(n)[pts >= elbow_val].max()
        if -1 <= offset <= 1:
            i_thres = max(0, min(i_thres + int(offset * i_thres), n - 1))
        else:
            i_thres = max(min(i_thres + int(offset), n - 1), 0)
        keep = np.zeros(n, dtype=bool)
        keep[i_thres:] = True
        return torch.from_numpy(keep).to(svals.device)

    @torch.no_grad()
    def get_eigens(self, fea_in, distinguisher=None):
        """Spectrum + basis of every protected layer's covariance (:360-380).

        The layers are independent d x d problems: under ``torch.distributed`` they are
        sharded over the ranks (owner by descending d^3, ``dist.shard_by_cost``), every owner
        runs cuSOLVER syevd on its layers and one broadcast per owner hands the results to
        everybody - the reference runs all of them on every rank, twice (SURVEY.md 8e)."""
        from . import dist as D
        jobs = []
        for group in self.param_groups:
            if group["svd"] is False:
                continue
            for n, p in zip(group["names"], group["params"]):
                if n not in fea_in.keys():
                    continue
                _lib.require_cuda(fea_in[n], "covariance of %s" % n)
                jobs.append(n)
        if not jobs:
            return

        def eig(i):
            cov = fea_in[jobs[i]]
            work = cov.to(self.eig_dtype)
            work = (work + work.t()) * 0.5
            evals, evecs = torch.linalg.eigh(work)          # cuSOLVER syevd
            order = torch.argsort(evals.abs(), descending=True)
            return evals.abs()[order].to(torch.float32), evecs[:, order].to(torch.float32)

        dims = [int(fea_in[n].shape[0]) for n in jobs]
        res = D.sharded_compute([((d,), (d, d)) for d in dims], [float(d) ** 3 for d in dims],
                                eig, fea_in[jobs[0]].device)
        for n, (vals, vecs) in zip(jobs, res):
            eigen = self.eigens[n]
            eigen["eigen_value"] = vals
            eigen["eigen_vector"] = vecs

    @torch.no_grad()
    def get_transforms(self, offset=0.0):
        """P = V0 V0^T over the null-side columns; 'backbone' names divided by
        ||P||_F (:235-290)."""
        for group in self.param_groups:
            if group["svd"] is False:
                continue
            for n, p in zip(group["names"], group["params"]):
                if n not in self.eigens.keys():
                    continue
                ind = self.adaptive_threshold(self.eigens[n]["eigen_value"], offset=offset)
                basis = self.eigens[n]["eigen_vector"][:, ind]
                transform = torch.mm(basis, basis.transpose(1, 0))
                scale = 1.0
                if "backbone" in n:
                    nrm = torch.norm(transform)
                    transform = transform / nrm
                    scale = 1.0 / float(nrm)
                self.transforms[n] = transform.detach()
                # the same projector in low-rank form: P = scale * (I - U U^T), U = the
                # kept-out (large-sigma) eigenvectors; used by step() while this tensor
                # stays in place and r is small
                kept_out = self.eigens[n]["eigen_vector"][:, ~ind].contiguous()
                self._lowrank[n] = (self.transforms[n], self.transforms[n]._version,
                                    kept_out, scale)

    # ---------------------------------------------------------------------- step
    def _prepare(self, name: str, P: torch.Tensor):
        key = (P.data_ptr(), P._version, tuple(P.shape))
        hit = self._prepared.get(name)
        if hit is not None and hit[0] == key:
            return hit[1], hit[2]
        _lib.require_cuda(P, "transform of %s" % name)
        if P.dim() != 2 or P.shape[0] != P.shape[1]:
            raise _lib.NsgpError("transform of %s must be square" % name)
        src = P.detach().float().contiguous()
        d = src.shape[0]
        ld = (d + 3) // 4 * 4
        hi = torch.empty(d, ld, dtype=torch.float32, device=P.device)
        lo = torch.empty_like(hi)
        check(lib.nsgp_projector_prepare(ptr(src), d, ptr(hi), ptr(lo),
                                         _lib.current_stream(P.device)),
              "nsgp_projector_prepare")
        self._prepared[name] = (key, hi, lo)
        return hi, lo

    def _prepare_lowrank(self, name: str, P: torch.Tensor):
        """(r, scale, ut_hi, ut_lo, un_hi, un_lo) when ``P`` is still the tensor that
        ``get_transforms`` built and its rank deficit is small, else None (dense form)."""
        lr = self._lowrank.get(name)
        if lr is None or lr[0] is not P or lr[1] != P._version:
            return None
        U, scale = lr[2], lr[3]
        d, r = U.shape
        if r == 0 or r > self.lowrank_max_ratio * d:
            return None
        hit = self._lowrank_prepared.get(name)
        if hit is not None and hit[0] is U:
            return hit[1]
        ld_d, ld_r = (d + 3) // 4 * 4, (r + 3) // 4 * 4
        ut_hi = torch.empty(r, ld_d, dtype=torch.float32, device=U.device)
        ut_lo = torch.empty_like(ut_hi)
        un_hi = torch.empty(d, ld_r, dtype=torch.float32, device=U.device)
        un_lo = torch.empty_like(un_hi)
        check(lib.nsgp_projector_prepare_lowrank(ptr(U), d, r, ptr(ut_hi), ptr(ut_lo),
                                                 ptr(un_hi), ptr(un_lo),
                                                 _lib.current_stream(U.device)),
              "nsgp_projector_prepare_lowrank")
        out = (r, scale, ut_hi, ut_lo, un_hi, un_lo)
        self._lowrank_prepared[name] = (U, out)
        return out

    def _staging(self, name: str, p: torch.Tensor):
        st = self._stage.get(name)
        cout = p.shape[0]
        need = cout * ((p.numel() // cout + 3) // 4 * 4)
        if st is None or st[0].numel() != need or st[0].device != p.device:
            st = (torch.empty(need, dtype=torch.float32, device=p.device),
                  torch.empty(need, dtype=torch.float32, device=p.device))
            self._stage[name] = st
        return st

    def _build_group_cache(self, gi, group, device, det):
        """Everything of a param group that survives from step to step: the ctypes tensor /
        layer tables, the T arena of its low-rank layers and the prepared plan.  Rebuilt when a
        parameter, a projector, the set of names or the deterministic mode (``det``, the plan's
        K-split partial tiles meet in a fixed order) changes."""
        names, params = group["names"], group["params"]
        n_t = len(params)
        tensors = (SgdTensor * n_t)()
        layers, t_need, protos = [], [], []
        svd = group["svd"]
        for i, (n, p) in enumerate(zip(names, params)):
            t = tensors[i]
            t.w, t.numel, t.layer = p.data_ptr(), p.numel(), -1
            if svd and len(self.transforms) > 0 and n in self.transforms.keys():
                P = self.transforms[n]
                cout = p.shape[0]
                dd = p.numel() // cout
                u_hi, u_lo = self._staging(n, p)
                low = self._prepare_lowrank(n, P)
                if low is None:
                    hi, lo = self._prepare(n, P)
                    L = ProjLayer(cout, dd, hi.data_ptr(), lo.data_ptr(),
                                  u_hi.data_ptr(), u_lo.data_ptr())
                else:
                    r, scale, ut_hi, ut_lo, un_hi, un_lo = low
                    L = ProjLayer(cout, dd, None, None, u_hi.data_ptr(), u_lo.data_ptr(),
                                  r, scale, ut_hi.data_ptr(), ut_lo.data_ptr(),
                                  un_hi.data_ptr(), un_lo.data_ptr())
                    t_need.append((len(layers), cout * ((r + 3) // 4 * 4)))
                t.layer = len(layers)
                layers.append(L)
                protos.append((n, P, P._version))
        # one arena [T | T_hi | T_lo] per group for its low-rank layers
        t_elems = sum(e for _, e in t_need)
        t_arena = None
        if t_elems:
            old = self._plans.get(gi)
            t_arena = old["t_arena"] if old is not None and old["t_arena"] is not None and \
                old["t_arena"].numel() == 3 * t_elems and old["t_arena"].device == device else \
                torch.empty(3 * t_elems, dtype=torch.float32, device=device)
            base, off = t_arena.data_ptr(), 0
            for li, e in t_need:
                layers[li].t = base + 4 * off
                layers[li].t_hi = base + 4 * (t_elems + off)
                layers[li].t_lo = base + 4 * (2 * t_elems + off)
                off += e
        n_l = len(layers)
        layer_arr = (ProjLayer * max(n_l, 1))(*layers)
        cache = dict(tensors=tensors, layer_arr=layer_arr, n_t=n_t, n_l=n_l, t_arena=t_arena,
                     t_elems=t_elems, protos=protos, w_ptrs=[p.data_ptr() for p in params],
                     g_ptrs=[0] * n_t, buf_ptrs=[0] * n_t, first=[-1] * n_t, plan=None,
                     buf=None, names=list(names), n_transforms=len(self.transforms),
                     uploaded=False, det=det)
        if _lib.engine() == 0:
            # ctypes fields read 0 until the first step fills g / buf; the plan only encodes the
            # weights, projectors and staging buffers
            need = int(lib.nsgp_sgd_plan_bytes(tensors, n_t, layer_arr, n_l))
            old = self._plans.get(gi)
            buf = old["buf"] if old is not None and old["buf"] is not None and \
                old["buf"].numel() >= need and old["buf"].device == device else \
                torch.empty(need, dtype=torch.uint8, device=device)
            plan = SgdPlan()
            check(lib.nsgp_sgd_plan_build(tensors, n_t, layer_arr, n_l, ptr(t_arena), t_elems,
                                          ptr(buf), buf.numel(), ctypes.byref(plan),
                                          _lib.current_stream(device)), "nsgp_sgd_plan_build")
            cache["plan"], cache["buf"] = plan, buf
        self._plans[gi] = cache
        return cache

    def _group_cache_valid(self, cache, group, det) -> bool:
        if cache is None or cache["names"] != group["names"] or \
                cache["n_transforms"] != len(self.transforms) or cache["det"] != det:
            return False
        for p, w in zip(group["params"], cache["w_ptrs"]):
            if p.data_ptr() != w:
                return False
        for n, P, ver in cache["protos"]:
            cur = self.transforms.get(n) if n in self.transforms.keys() else None
            if cur is not P or P._version != ver:
                return False
        return True

    @torch.no_grad()
    def step(self, closure=None):
        """One optimisation step (:59-96)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for gi, group in enumerate(self.param_groups):
            names, params = group["names"], group["params"]
            if len(params) == 0:
                continue
            device = params[0].device
            svd = group["svd"]
            # ---- validate everything before any state is touched
            grads = []
            for n, p in zip(names, params):
                grad = p.grad.data          # AttributeError when grad is None, like :75
                if grad.is_sparse:
                    raise RuntimeError("Adam does not support sparse gradients, please "
                                       "consider SparseAdam instead")
                _lib.require_cuda(p, "parameter %s" % n)
                if p.dtype != torch.float32 or grad.dtype != torch.float32 or \
                        not p.is_contiguous() or not grad.is_contiguous():
                    raise _lib.NsgpError("parameter %s: fp32 contiguous tensors required" % n)
                if svd and len(self.transforms) > 0 and n in self.transforms.keys():
                    if p.dim() not in (2, 4):
                        raise _lib.NsgpError("parameter %s: projection needs a 2-D or 4-D "
                                             "tensor" % n)
                    P = self.transforms[n]
                    cout = p.shape[0]
                    dd = p.numel() // cout
                    if P.shape[0] != dd:
                        raise RuntimeError("mat1 and mat2 shapes cannot be multiplied "
                                           "(%dx%d and %dx%d)" % (cout, dd, P.shape[0], P.shape[1]))
                grads.append(grad)
            det = _lib.deterministic()
            cache = self._plans.get(gi)
            if not self._group_cache_valid(cache, group, det):
                cache = self._build_group_cache(gi, group, device, det)
            tensors = cache["tensors"]
            changed = not cache["uploaded"]
            g_ptrs, buf_ptrs, first = cache["g_ptrs"], cache["buf_ptrs"], cache["first"]
            for i, (p, grad) in enumerate(zip(params, grads)):
                state = self.state[p]
                if len(state) == 0:
                    state["step"] = 0
                    state["previous_grad"] = torch.zeros_like(p.data)
                state["step"] += 1
                f = 1 if state["step"] == 1 else 0
                gp, bp = grad.data_ptr(), state["previous_grad"].data_ptr()
                if gp != g_ptrs[i] or bp != buf_ptrs[i] or f != first[i]:
                    t = tensors[i]
                    t.g, t.buf, t.first_step = gp, bp, f
                    g_ptrs[i], buf_ptrs[i], first[i] = gp, bp, f
                    changed = True
            stream = _lib.current_stream(device)
            hyper = (float(group["lr"]), float(group["momentum"]), float(group["dampening"]),
                     float(group["weight_decay"]), 1 if group["nesterov"] else 0)
            n_t, n_l, layer_arr = cache["n_t"], cache["n_l"], cache["layer_arr"]
            if cache["plan"] is None:
                # bring-up engine: one-shot call, per-layer launches
                need = lib.nsgp_sgd_step_workspace_bytes(n_t, n_l)
                if self._workspace is None or self._workspace.numel() < need or \
                        self._workspace.device != device:
                    self._workspace = torch.empty(int(need), dtype=torch.uint8, device=device)
                check(lib.nsgp_sgd_nscl_step(tensors, n_t, layer_arr, n_l, *hyper,
                                             ptr(self._workspace), self._workspace.numel(),
                                             stream), "nsgp_sgd_nscl_step")
                continue
            # the tensor table travels only when a gradient / momentum pointer or a first-step
            # flag changed since the last upload
            check(lib.nsgp_sgd_plan_step(tensors if changed else None, n_t, layer_arr, n_l,
                                         ptr(cache["buf"]), ctypes.byref(cache["plan"]), *hyper,
                                         stream), "nsgp_sgd_plan_step")
            cache["uploaded"] = True
        return loss
