"""RoIAlign 256x7x7 extraction over the FPN levels (SURVEY.md 8f-2) - drop-in for
``SingleRoIExtractor`` (mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py)
with ``roi_layer=dict(type='RoIAlign', output_size=7, sampling_ratio=0)`` and
``featmap_strides=[4, 8, 16, 32]`` (cl_faster_rcnn_nsgp_repre_19_1_2.py:72-75).

The reference maps RoIs to levels, then per level gathers the RoIs (``nonzero``: a host
sync per level), calls mmcv's RoIAlign and scatters the result back.  Here ONE launch
handles all levels, and ``class_sums`` adds the features straight into the per-class sums
of the coarse prototypes (standard_roi_replay_head.py:411-415) without writing the
(R, 12544) feature matrix.

Differentiable w.r.t. the feature maps (``repre_roi_align_backward``: the transpose of the
pooling, atomics into zero-filled gradient maps), so it serves the training forward of the
RoI head as well as the no-grad paths (``get_bbox_stuff`` during ``cal_rois``,
nsrunner_roi_replay.py:776-868, and the teacher's ``predict``).  Like mmcv's op it has no
gradient w.r.t. the RoI coordinates.
"""
from __future__ import annotations

import ctypes

import torch
import torch.nn as nn

from . import _lib
from ._lib import lib, check, ptr


class _RoIAlignFn(torch.autograd.Function):
    """forward = the multi-level launch; backward = its transpose into fresh gradient maps."""

    @staticmethod
    def forward(ctx, ext, rois, levels, *feats):
        with torch.no_grad():
            out, _, _, (C, P) = ext._launch(feats, rois, None, None, 0, True, levels)
        ctx.ext = ext
        ctx.levels = levels
        ctx.shapes = [tuple(f.shape) for f in feats]
        ctx.save_for_backward(rois)
        return out.view(-1, C, P, P)

    @staticmethod
    def backward(ctx, grad_out):
        ext = ctx.ext
        (rois,) = ctx.saved_tensors
        dev = grad_out.device
        # the transpose scatters with atomicAdd (as torchvision's roi_align backward does)
        _lib.alert_not_deterministic("repre_roi_align_backward")
        L = len(ctx.shapes)
        grads = [torch.zeros(sh, dtype=torch.float32, device=dev) for sh in ctx.shapes]
        R = rois.shape[0]
        if R > 0:
            B, C = ctx.shapes[0][0], ctx.shapes[0][1]
            go = grad_out.detach().float().contiguous()
            r = rois.detach().float().contiguous()
            ptrs = (ctypes.c_void_p * L)(*[g.data_ptr() for g in grads])
            hs = (ctypes.c_int32 * L)(*[sh[2] for sh in ctx.shapes])
            ws = (ctypes.c_int32 * L)(*[sh[3] for sh in ctx.shapes])
            sc = (ctypes.c_float * L)(*[1.0 / s for s in ext.featmap_strides[:L]])
            check(lib.repre_roi_align_backward(ptrs, hs, ws, sc, L, B, C, ptr(r), R,
                                               ext.output_size, ext.sampling_ratio,
                                               1 if ext.aligned else 0, float(ext.finest_scale),
                                               ptr(ctx.levels), ptr(go), _lib.current_stream(dev)),
                  "repre_roi_align_backward")
        return (None, None, None) + tuple(grads)


class SingleRoIExtractor(nn.Module):
    """Constructor keywords of the reference (:32-43); ``roi_layer`` accepts the mmcv
    config dict (``type='RoIAlign'``, ``output_size``, ``sampling_ratio``, ``aligned``,
    ``pool_mode='avg'``)."""

    def __init__(self, roi_layer: dict, out_channels: int, featmap_strides, finest_scale: int = 56,
                 init_cfg=None):
        super().__init__()
        cfg = dict(roi_layer)
        typ = cfg.pop("type", "RoIAlign")
        if typ != "RoIAlign":
            raise _lib.NsgpError("only roi_layer type 'RoIAlign' is implemented (got %r)" % (typ,))
        if cfg.get("pool_mode", "avg") != "avg":
            raise _lib.NsgpError("RoIAlign pool_mode must be 'avg'")
        osz = cfg.get("output_size", 7)
        if isinstance(osz, (tuple, list)):
            if osz[0] != osz[1]:
                raise _lib.NsgpError("RoIAlign output_size must be square")
            osz = osz[0]
        self.output_size = int(osz)
        self.sampling_ratio = int(cfg.get("sampling_ratio", 0))
        self.aligned = bool(cfg.get("aligned", True))
        self.out_channels = out_channels
        self.featmap_strides = list(featmap_strides)
        self.finest_scale = finest_scale

    @property
    def num_inputs(self) -> int:
        return len(self.featmap_strides)

    def map_roi_levels(self, rois: torch.Tensor, num_levels: int) -> torch.Tensor:
        """:45-63 (torch ops; the kernel evaluates the same expression per RoI)."""
        scale = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
        target_lvls = torch.floor(torch.log2(scale / self.finest_scale + 1e-6))
        return target_lvls.clamp(min=0, max=num_levels - 1).long()

    @staticmethod
    def roi_rescale(rois: torch.Tensor, scale_factor: float) -> torch.Tensor:
        """base_roi_extractor.py:70-92."""
        cx = (rois[:, 1] + rois[:, 3]) * 0.5
        cy = (rois[:, 2] + rois[:, 4]) * 0.5
        w = rois[:, 3] - rois[:, 1]
        h = rois[:, 4] - rois[:, 2]
        new_w, new_h = w * scale_factor, h * scale_factor
        return torch.stack((rois[:, 0], cx - new_w * 0.5, cy - new_h * 0.5, cx + new_w * 0.5,
                            cy + new_h * 0.5), dim=-1)

    def _launch(self, feats, rois, roi_scale_factor, labels, num_classes, want_feats,
                levels=None):
        feats = list(feats)[: self.num_inputs]
        f0 = feats[0]
        _lib.require_cuda(f0, "feature maps")
        rois = rois.type_as(f0)                                                  # :81
        if roi_scale_factor is not None:
            # :96-99 - the level comes from the unscaled RoI, then the RoI is rescaled
            if len(feats) > 1:
                levels = self.map_roi_levels(rois, len(feats)).to(torch.int32).contiguous()
            rois = self.roi_rescale(rois, roi_scale_factor)
        L = len(feats)
        B, C = f0.shape[0], f0.shape[1]
        fs = []
        for f in feats:
            if f.dtype != torch.float32 or not f.is_contiguous():
                f = f.float().contiguous()
            fs.append(f)
        rois = rois.float().contiguous()
        R = rois.shape[0]
        P = self.output_size
        D = C * P * P
        ptrs = (ctypes.c_void_p * L)(*[f.data_ptr() for f in fs])
        hs = (ctypes.c_int32 * L)(*[f.shape[2] for f in fs])
        ws = (ctypes.c_int32 * L)(*[f.shape[3] for f in fs])
        sc = (ctypes.c_float * L)(*[1.0 / s for s in self.featmap_strides[:L]])
        out = torch.empty(R, D, dtype=torch.float32, device=f0.device) if want_feats else None
        sums = counts = None
        if labels is not None:
            labels = labels.to(device=f0.device, dtype=torch.int64).contiguous()
            sums = torch.empty(num_classes, D, dtype=torch.float32, device=f0.device)
            counts = torch.empty(num_classes, dtype=torch.int32, device=f0.device)
        if R == 0:                      # :91-92 - nothing to pool (an empty tensor has no address)
            if sums is not None:
                sums.zero_()
                counts.zero_()
            return out, sums, counts, (C, P)
        check(lib.repre_roi_align(ptrs, hs, ws, sc, L, B, C, ptr(rois), R, P, self.sampling_ratio,
                                  1 if self.aligned else 0, float(self.finest_scale),
                                  ptr(levels), ptr(labels), int(num_classes or 0), ptr(out), ptr(sums),
                                  ptr(counts), _lib.current_stream(f0.device)),
              "repre_roi_align")
        return out, sums, counts, (C, P)

    def forward(self, feats, rois, roi_scale_factor=None):
        """:65-118 - (R, out_channels, 7, 7) RoI features."""
        feats = list(feats)[: self.num_inputs]
        if torch.is_grad_enabled() and any(f.requires_grad for f in feats):
            levels = None
            rois = rois.type_as(feats[0]).detach()
            if roi_scale_factor is not None:
                if len(feats) > 1:
                    levels = self.map_roi_levels(rois, len(feats)).to(torch.int32).contiguous()
                rois = self.roi_rescale(rois, roi_scale_factor)
            fs = [f if f.dtype == torch.float32 and f.is_contiguous() else f.float().contiguous()
                  for f in feats]
            _lib.require_cuda(fs[0], "feature maps")
            return _RoIAlignFn.apply(self, rois, levels, *fs)
        with torch.no_grad():
            out, _, _, (C, P) = self._launch(feats, rois, roi_scale_factor, None, 0, True)
        return out.view(-1, C, P, P)

    @torch.no_grad()
    def class_sums(self, feats, rois, labels, num_classes, return_feats=False):
        """RoIAlign fused with the per-class sums: returns (sums (num_classes, C*7*7),
        counts (num_classes,) int32[, feats (R, C*7*7)]); ``sums / counts`` are the coarse
        prototypes ``mean(F[label == c], 0)`` of standard_roi_replay_head.py:411-415.  The sums
        are atomicAdd'ed: raises (warns) under ``torch.use_deterministic_algorithms(True)``."""
        _lib.alert_not_deterministic("SingleRoIExtractor.class_sums")
        out, sums, counts, _ = self._launch(feats, rois, None, labels, num_classes, return_feats)
        return (sums, counts, out) if return_feats else (sums, counts)


def reduce_class_sums(sums: torch.Tensor, counts: torch.Tensor, group=None):
    """Data-parallel coarse prototypes (SURVEY 8e): every rank pools its own RoIs into per-class
    sums / counts (``SingleRoIExtractor.class_sums``), ONE all-reduce of the (C, D) sums and
    the (C,) counts makes them global - no RoI feature ever crosses the fabric - and
    ``sums / counts`` is ``mean(F[label == c], 0)`` over the RoIs of all ranks
    (standard_roi_replay_head.py:411-415).  Classes without RoIs come back as NaN like
    ``torch.mean`` of an empty slice.  Returns (means (C, D), counts (C,) int64)."""
    import torch.distributed as dist
    counts = counts.to(torch.int64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        w1 = dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group, async_op=True)
        w2 = dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group, async_op=True)
        w1.wait()
        w2.wait()
    return sums / counts.to(sums.dtype).unsqueeze(1), counts
