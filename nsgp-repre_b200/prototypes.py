"""RePRE prototype build + replay staging, drop-in for
``StandardMultiPrototypeReplayHead`` (mmdet/models/roi_heads/
standard_roi_replay_head.py:375-501).

Everything runs on the device - the stable class index (the boolean-mask gather of :412),
per-class segmented means (:412-414), L2-normalise + cosine Gram + ``>= 0.6`` + neighbour
counts (:417-421), the density ordering and the greedy cover (:421-448: one CTA per class; a
stable descending rank reproduces the tie order of torch's CPU sort), masked means (:443),
the device-resident replay gather (:458-463).  The build is a FIXED sequence of launches
sized from the number of rows M: no class size is read back in the middle; the host reads a
few bytes once at the end (number of prototypes, status) and ``save_idx`` (the ``mask.pth``
payload) only when it is asked for.
"""
from __future__ import annotations

import os
import os.path as osp

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from ._lib import lib, check, ptr


def get_work_dir(previous_path: str) -> str:
    """Path rule of :363-370: '..._N' -> '..._N+1' ('coco' paths -> './')."""
    if "coco" in previous_path:
        return "./"
    parts = previous_path.split("_")
    parts[-1] = str(int(parts[-1]) + 1)
    return "_".join(parts)


class MultiPrototypeReplay:
    """Builds and serves the coarse + fine-grained prototypes of the old classes.

    ``build`` mirrors the loop at :404-449; results: ``bbox_featss`` (P,D) fp32 on
    the device, ``tmp_label`` (P,) int64, ``save_idx`` = the ``mask.pth`` payload
    (list[class] of list[<=max_proto-1] bool masks over that class's rows).
    """

    def __init__(self, max_prototype: int = 10, thresh: float = 0.6):
        self.max_proto = max_prototype
        self.thresh = thresh
        self.bbox_featss = None
        self.tmp_label = None
        self._save_idx = None
        self._lazy_masks = None
        self.sigma = None
        self._out = None
        self._ws = None
        self._bufs = None
        self._segments = None
        self._graph = None          # (key, torch.cuda.CUDAGraph) of a repeated build
        self._graph_seen = None
        self.use_graph = True

    # ------------------------------------------------------------------ build
    @torch.no_grad()
    def build(self, feats: torch.Tensor, cls_targets: torch.Tensor, previous_cls,
              saved_masks=None):
        _lib.require_cuda(feats, "bbox_featss")
        dev = feats.device
        feats = feats.detach()
        feats = feats.reshape(feats.shape[0], -1)
        if feats.dtype != torch.float32 or not feats.is_contiguous():
            feats = feats.float().contiguous()
        M, D = feats.shape
        labels = cls_targets.detach().to(device=dev, dtype=torch.int64).contiguous()
        previous_cls = list(previous_cls)
        save_idx = list(saved_masks) if saved_masks is not None else []
        if not previous_cls:
            self.bbox_featss = feats.new_zeros(0, D)
            self.tmp_label = torch.zeros(0, dtype=torch.long, device=dev)
            self.save_idx = save_idx
            return self

        if M == 0:
            raise IndexError("class %d has no stored RoI feature "
                             "(index 0 is out of bounds for dimension 0 with size 0)"
                             % previous_cls[0])
        consecutive = all(b == a + 1 for a, b in zip(previous_cls, previous_cls[1:]))
        if not consecutive:
            # the reference always passes range(...); an arbitrary class list is built class
            # run by class run and concatenated
            parts, start = [], 0
            for i in range(1, len(previous_cls) + 1):
                if i == len(previous_cls) or previous_cls[i] != previous_cls[i - 1] + 1:
                    parts.append(previous_cls[start:i])
                    start = i
            subs = [MultiPrototypeReplay(self.max_proto, self.thresh).build(
                feats, labels, p, saved_masks) for p in parts]
            self.bbox_featss = torch.cat([m.bbox_featss for m in subs])
            self.tmp_label = torch.cat([m.tmp_label for m in subs])
            # the runs in order walk previous_cls in order, as the reference's loop does
            merged = list(save_idx)
            for m in subs:
                _place_masks(merged, m._class_masks())
            self.save_idx = merged
            self._segments, self._feats = None, feats
            return self
        return self._build_device(feats, labels, M, D, previous_cls, save_idx)

    def _build_device(self, feats, labels, M, D, previous_cls, saved_masks):
        """The stable class index (one launch) and everything after it as ONE C-ABI call
        (``repre_build_prototypes``): a fixed sequence of launches sized from M - no class size
        is read back; the host reads a few bytes at the end (number of prototypes, status)
        and the masks lazily.  A build repeated on the same input buffers (same addresses and
        shapes, no replayed masks) replays a CUDA graph of that sequence from its third run on."""
        import ctypes
        dev = feats.device
        ncls = len(previous_cls)
        c0 = previous_cls[0]
        C = previous_cls[-1] + 1
        mp = self.max_proto - 1
        # deterministic mode: the Gram's K-split partial tiles meet in split order and the
        # segment means are one sequential pass per segment; the workspace (and a recorded
        # graph) belongs to one mode
        det = _lib.deterministic()
        need = int(lib.repre_build_prototypes_workspace_bytes(M, D, ncls, mp))
        key = (M, D, C, ncls, mp, dev, det)
        if self._bufs is None or self._bufs[0] != key:
            nseg_max = ncls * (mp + 1)
            self._bufs = (key, dict(
                ws=torch.empty(need, dtype=torch.uint8, device=dev),
                cls_counts=torch.empty(C, dtype=torch.int32, device=dev),
                offsets=torch.empty(C + 1, dtype=torch.int32, device=dev),
                rows=torch.empty(M, dtype=torch.int32, device=dev),
                masks=torch.empty(M * M, dtype=torch.uint8, device=dev),
                counts=torch.empty(M, dtype=torch.int32, device=dev),
                seg_off=torch.empty(nseg_max + 1, dtype=torch.int32, device=dev),
                seg_rows=torch.empty(M * (mp + 1), dtype=torch.int32, device=dev),
                seg_label=torch.empty(nseg_max, dtype=torch.int32, device=dev),
                info=torch.empty(1 + ncls + ncls * mp + 2, dtype=torch.int32, device=dev),
                out=torch.empty(nseg_max, D, dtype=torch.float32, device=dev)))
            self._graph, self._graph_seen = None, None
        b = self._bufs[1]
        # masks replayed from mask.pth (:425-433): one H2D of the packed bytes
        saved_dev, n_saved_arr, len_arr = None, None, None
        saved_lists = [list(saved_masks[c]) if c < len(saved_masks) else [] for c in previous_cls]
        if any(saved_lists):
            n_saved = [min(len(l), mp) for l in saved_lists]
            lens = [int(l[0].numel()) if l else 0 for l in saved_lists]
            chunks = []
            for l, k, n in zip(saved_lists, n_saved, lens):
                for m in l[:k]:
                    if m.numel() != n:
                        raise IndexError("replayed masks of one class differ in length")
                    chunks.append(m.cpu().to(torch.uint8).reshape(-1))
            if chunks:
                saved_dev = torch.cat(chunks).to(dev)
                n_saved_arr = (ctypes.c_int32 * ncls)(*n_saved)
                len_arr = (ctypes.c_int32 * ncls)(*lens)

        def launch(flags):
            stream = _lib.current_stream(dev)
            check(lib.repre_class_index(ptr(labels), M, C, ptr(b["cls_counts"]),
                                        ptr(b["offsets"]), ptr(b["rows"]), stream),
                  "repre_class_index")
            check(lib.repre_build_prototypes(
                ptr(feats), D, M, ptr(b["rows"]), ptr(b["offsets"]), c0, ncls,
                float(self.thresh), mp, ptr(saved_dev), n_saved_arr, len_arr, ptr(b["masks"]),
                ptr(b["counts"]), ptr(b["seg_off"]), ptr(b["seg_rows"]), ptr(b["seg_label"]),
                ptr(b["info"]), ptr(b["out"]), ptr(b["ws"]), b["ws"].numel(), flags, stream),
                "repre_build_prototypes")

        gkey = (feats.data_ptr(), labels.data_ptr(), c0, float(self.thresh))
        graph_ok = self.use_graph and saved_dev is None and not _lib.PROFILE_ON
        if graph_ok and self._graph is not None and self._graph[0] == gkey:
            self._graph[1].replay()
        else:
            launch(0)
            if graph_ok and self._graph_seen == gkey:
                # second build on the same buffers: record the launch sequence (the tables of
                # the first call are still in the workspace) for the following ones
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    launch(1)
                self._graph = (gkey, g)
            self._graph_seen = gkey if graph_ok else None
        counts = b["cls_counts"]
        h_info = b["info"].cpu().tolist()                             # the one (late) sync
        nseg, status = h_info[0], h_info[1 + ncls + ncls * mp]
        if status == 1:
            # the reference dies in sim_sum[-0//3] (:422); keep that contract
            h_cnt = counts.cpu().tolist()
            empty = [c for c in previous_cls if h_cnt[c] == 0]
            raise IndexError("class %d has no stored RoI feature "
                             "(index 0 is out of bounds for dimension 0 with size 0)" % empty[0])
        if status == 2:
            raise IndexError("a replayed mask does not have one entry per row of its class "
                             "(The shape of the mask does not match the tensor)")
        self.bbox_featss = b["out"][:nseg]
        self.tmp_label = b["seg_label"][:nseg].to(torch.int64)
        self._segments = (b["seg_off"], b["seg_rows"], M)
        self._feats = feats
        self._lazy_masks = (b["masks"], counts, list(previous_cls), h_info[1:1 + ncls],
                            h_info[1 + ncls:1 + ncls + ncls * mp], saved_lists,
                            list(saved_masks), mp)
        self._save_idx = None
        return self

    @property
    def save_idx(self):
        """``mask.pth`` payload (:450-452): list[class] of list of bool masks over the
        class's rows; built from the device picks on first access."""
        if self._save_idx is None and self._lazy_masks is not None:
            save_idx = self._lazy_masks[6]
            self._save_idx = _place_masks(save_idx, self._class_masks())
            self._lazy_masks = None
        return self._save_idx

    def _class_masks(self):
        """[(class, masks)] of the last device build in class order: a class's replayed masks
        followed by the masks of its new picks."""
        masks, counts, classes, npicks, picks, saved_lists, _, mp = self._lazy_masks
        h_cnt = counts.cpu().tolist()
        out, moff = [], 0
        for ci, c in enumerate(classes):
            n = h_cnt[c]
            tmp = list(saved_lists[ci])
            mine = [p for p in picks[ci * mp:ci * mp + npicks[ci]] if p >= 0]
            if mine:
                idx = torch.tensor(mine, dtype=torch.int64, device=masks.device)
                sel = masks[moff:moff + n * n].view(n, n)[idx].cpu().bool()
                tmp.extend(sel[k].clone() for k in range(len(mine)))
            moff += n * n
            out.append((c, tmp))
        return out

    @save_idx.setter
    def save_idx(self, value):
        self._save_idx = value
        self._lazy_masks = None

    @torch.no_grad()
    def build_sigma(self):
        """Extension (BASELINE north_star item 4; no reference counterpart): per-
        prototype diagonal standard deviation for Gaussian replay."""
        off_t, all_rows, max_rows = self._segments
        nseg, D = self.bbox_featss.shape
        var = torch.empty_like(self.bbox_featss)
        _lib.deterministic()
        check(lib.repre_segment_var(ptr(self._feats), D, ptr(off_t), ptr(all_rows), nseg,
                                    int(max_rows), ptr(self.bbox_featss), ptr(var),
                                    _lib.current_stream(var.device)), "repre_segment_var")
        self.sigma = var.sqrt_()
        return self.sigma

    # ----------------------------------------------------------------- replay
    @torch.no_grad()
    def staged(self, idx=None, out=None, sigma=None, seed=0):
        """Classifier input of the replay branch (:458-463): the prototypes are
        device-resident; this gathers them (all of them when ``idx`` is None, as
        the reference stages every prototype every step) into ``out``."""
        protos = self.bbox_featss
        P = protos.shape[0] if idx is None else idx.shape[0]
        D = protos.shape[1]
        if out is None:
            if self._out is None or self._out.shape != (P, D):
                self._out = torch.empty(P, D, dtype=torch.float32, device=protos.device)
            out = self._out
        if idx is not None:
            idx = idx.to(device=protos.device, dtype=torch.int64).contiguous()
        check(lib.repre_replay_gather(ptr(protos), ptr(sigma), ptr(idx), P, D, int(seed),
                                      ptr(out), _lib.current_stream(protos.device)),
              "repre_replay_gather")
        return out


def _place_masks(save_idx, class_masks):
    """The ``mask.pth`` rule of :425-452 over ``(class, masks)`` in class order: a class below
    ``len(save_idx)`` replaces its entry, any other class is appended."""
    for c, masks in class_masks:
        if c < len(save_idx):
            save_idx[c] = masks
        else:
            save_idx.append(masks)
    return save_idx


def exchange_by_class_owner(feats, labels, classes, group=None):
    """The one exchange step of a data-parallel prototype build (SURVEY.md 8e): class ``c``
    is owned by rank ``classes.index(c) % W``; every rank sends the rows of each class to its
    owner.  Returns ``(feats_owned, labels_owned, owned_classes)``; rows arrive in (source
    rank, original row) order, i.e. the order they have in the reference's gathered
    ``rois_etc.pth`` (``cat(all_gather_different_shape(...))``, nsrunner_roi_replay.py:815-820),
    so neighbour masks and tie orders equal the single-process build."""
    import torch.distributed as dist
    classes = list(classes)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return feats, labels, classes
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    owner_of = torch.full((max(classes) + 2,), -1, dtype=torch.int64, device=labels.device)
    for k, c in enumerate(classes):
        owner_of[c] = k % world
    lab = labels.to(torch.int64)
    own = torch.where((lab >= 0) & (lab <= max(classes)), owner_of[lab.clamp(0, max(classes))],
                      torch.full_like(lab, -1))
    order = torch.argsort(own, stable=True)               # by destination, original order kept
    order = order[own[order] >= 0]
    send_counts = torch.bincount(own[order], minlength=world)[:world]
    recv_counts = torch.empty_like(send_counts)
    dist.all_to_all_single(recv_counts, send_counts, group=group) \
        if dist.get_backend(group) == "nccl" else _gloo_counts(recv_counts, send_counts, group)
    sc, rc = send_counts.tolist(), recv_counts.tolist()
    send_f = feats.reshape(feats.shape[0], -1)[order].contiguous()
    send_l = lab[order].contiguous()
    recv_f = send_f.new_empty((sum(rc), send_f.shape[1]))
    recv_l = send_l.new_empty((sum(rc),))
    if dist.get_backend(group) == "nccl":
        dist.all_to_all_single(recv_f, send_f, rc, sc, group=group)
        dist.all_to_all_single(recv_l, send_l, rc, sc, group=group)
    else:                                                  # gloo (CPU tests): var-len gathers
        from .rois import all_gather_different_shape
        offs = [0]
        for n in sc:
            offs.append(offs[-1] + n)
        f_parts, l_parts = [], []
        for dst in range(world):
            fp = all_gather_different_shape(send_f[offs[dst]:offs[dst + 1]], group)
            lp = all_gather_different_shape(send_l[offs[dst]:offs[dst + 1]], group)
            if dst == rank:
                f_parts, l_parts = fp, lp
        recv_f, recv_l = torch.cat(f_parts), torch.cat(l_parts)
    owned = [c for k, c in enumerate(classes) if k % world == rank]
    return recv_f, recv_l, owned


def _gloo_counts(recv_counts, send_counts, group):
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    table = [torch.empty_like(send_counts) for _ in range(world)]
    dist.all_gather(table, send_counts, group=group)
    for src in range(world):
        recv_counts[src] = table[src][rank]


def gather_prototypes(protos, tmp_label, group=None):
    """All ranks' prototypes in the reference order (classes ascending, coarse prototype
    first, then the fine ones in pick order): var-len all-gather + stable sort by class."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return protos, tmp_label
    from .rois import all_gather_different_shape
    p_all = torch.cat(all_gather_different_shape(protos, group))
    l_all = torch.cat(all_gather_different_shape(tmp_label, group))
    order = torch.argsort(l_all, stable=True)
    return p_all[order].contiguous(), l_all[order].contiguous()


@torch.no_grad()
def build_prototypes_sharded(feats, cls_targets, previous_cls, max_prototype=10, group=None):
    """Data-parallel form of the prototype build: every rank passes the RoI features it
    harvested; classes are sharded over the ranks (one all-to-all of the foreground rows),
    each owner runs the device build for its classes, the (<= 20 MB of) prototypes are
    all-gathered.  Returns a ``MultiPrototypeReplay`` holding all prototypes on every rank."""
    f_own, l_own, owned = exchange_by_class_owner(feats, cls_targets, previous_cls, group)
    mp = MultiPrototypeReplay(max_prototype).build(f_own, l_own, owned)
    protos, labels = gather_prototypes(mp.bbox_featss, mp.tmp_label, group)
    out = MultiPrototypeReplay(max_prototype)
    out.bbox_featss, out.tmp_label = protos, labels
    out.local = mp                     # this rank's classes: masks / segments for mask.pth
    return out


@torch.no_grad()
def kmeans_prototypes(feats: torch.Tensor, init_centres: torch.Tensor, iters: int = 10):
    """Extension (BASELINE north_star item 3; the reference imports sklearn's KMeans at
    standard_roi_replay_head.py:18 and never calls it - parity unpinned, checked against
    ``oracle.restated.kmeans_assign / kmeans_update``): Lloyd iterations from explicit
    initial centres, entirely on the device.  Assignment = argmin_k |x - c_k|^2 (ties ->
    lowest k) through the tcgen05 contraction X C^T, update = segmented mean of the rows of
    every cluster (an empty cluster keeps its centre).  Returns (centres (k,D), labels (n,))."""
    _lib.require_cuda(feats, "features")
    _lib.alert_not_deterministic("kmeans_prototypes")
    _lib.deterministic()
    dev = feats.device
    x = feats.detach().reshape(feats.shape[0], -1)
    if x.dtype != torch.float32 or not x.is_contiguous():
        x = x.float().contiguous()
    n, D = x.shape
    centres = init_centres.detach().to(device=dev, dtype=torch.float32).reshape(-1, D).clone()
    k = centres.shape[0]
    stream = _lib.current_stream(dev)
    ws = torch.empty(int(lib.repre_kmeans_assign_workspace_bytes(n, k, D)), dtype=torch.uint8,
                     device=dev)
    labels = torch.empty(n, dtype=torch.int64, device=dev)
    counts = torch.empty(k, dtype=torch.int32, device=dev)
    offsets = torch.empty(k + 1, dtype=torch.int32, device=dev)
    rows = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    new = torch.empty_like(centres)
    for _ in range(max(1, int(iters))):
        check(lib.repre_kmeans_assign(ptr(x), n, D, ptr(centres), k, ptr(labels), ptr(ws),
                                      ws.numel(), stream), "repre_kmeans_assign")
        check(lib.repre_class_index(ptr(labels), n, k, ptr(counts), ptr(offsets), ptr(rows),
                                    stream), "repre_class_index")
        check(lib.repre_segment_mean(ptr(x), D, ptr(offsets), ptr(rows), k, n, ptr(new), stream),
              "repre_segment_mean")
        centres = torch.where((counts > 0).unsqueeze(1), new, centres)
    check(lib.repre_kmeans_assign(ptr(x), n, D, ptr(centres), k, ptr(labels), ptr(ws),
                                  ws.numel(), stream), "repre_kmeans_assign")
    return centres, labels


class SampledRoIReplay:
    """Device-resident store of ``rois_etc.pth`` and the sampled gather of
    ``StandardRoIReplayHead.loss`` (standard_roi_replay_head.py:53-69): the reference keeps
    the six tensors wherever ``torch.load`` put them, indexes all six with
    ``randperm(M)[:64]`` and moves the 64 rows to the model's device every step (3.2 MB
    pageable H2D).  Here the six tensors live on the device, the 64 indices (512 B) are the
    only H2D traffic and ONE launch gathers all six (``repre_replay_gather_rois``).  The
    indices are drawn exactly like the reference (``torch.randperm`` on the default CPU
    generator), so a seeded run replays the same RoIs."""

    FIELDS = ("bbox_featss", "cls_targets", "cls_weights", "bbox_targets", "bbox_weights",
              "roiss")

    def __init__(self, tensors, device=None, sample_size=64):
        if len(tensors) != 6:
            raise ValueError("rois_etc.pth holds a list of 6 tensors")
        dev = torch.device(device) if device is not None else torch.device("cuda")
        f, ct, cw, bt, bw, r = tensors
        M = f.shape[0]
        self.bbox_featss = f.detach().reshape(M, -1).to(dev, torch.float32).contiguous()
        self.cls_targets = ct.detach().reshape(M).to(dev, torch.int64).contiguous()
        self.cls_weights = cw.detach().reshape(M).to(dev, torch.float32).contiguous()
        self.bbox_targets = bt.detach().reshape(M, 4).to(dev, torch.float32).contiguous()
        self.bbox_weights = bw.detach().reshape(M, 4).to(dev, torch.float32).contiguous()
        self.roiss = r.detach().reshape(M, 5).to(dev, torch.float32).contiguous()
        _lib.require_cuda(self.bbox_featss, "rois_etc.pth tensors")
        self.sample_size = sample_size
        self._out = None

    @classmethod
    def load(cls, previous_path, device=None, **kw):
        return cls(torch.load(osp.join(previous_path, "rois_etc.pth"), map_location="cpu"),
                   device=device, **kw)

    @torch.no_grad()
    def sample(self, idx=None):
        """(bbox_featss, cls_targets, cls_weights, bbox_targets, bbox_weights, roiss) at
        ``idx`` (default ``torch.randperm(M)[:64]``, :58)."""
        M, D = self.bbox_featss.shape
        if idx is None:
            idx = torch.randperm(M)[:self.sample_size]
        dev = self.bbox_featss.device
        idx = idx.to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        P = idx.shape[0]
        if self._out is None or self._out[0].shape[0] != P:
            self._out = (torch.empty(P, D, dtype=torch.float32, device=dev),
                         torch.empty(P, dtype=torch.int64, device=dev),
                         torch.empty(P, dtype=torch.float32, device=dev),
                         torch.empty(P, 4, dtype=torch.float32, device=dev),
                         torch.empty(P, 4, dtype=torch.float32, device=dev),
                         torch.empty(P, 5, dtype=torch.float32, device=dev))
        o = self._out
        check(lib.repre_replay_gather_rois(
            ptr(self.bbox_featss), ptr(self.cls_targets), ptr(self.cls_weights),
            ptr(self.bbox_targets), ptr(self.bbox_weights), ptr(self.roiss), ptr(idx), P, D,
            ptr(o[0]), ptr(o[1]), ptr(o[2]), ptr(o[3]), ptr(o[4]), ptr(o[5]),
            _lib.current_stream(dev)), "repre_replay_gather_rois")
        return o


class ReplayHeadMixin:
    """The replay logic of both reference heads, written once and bound onto whatever
    ``StandardRoIHead`` is available (mmdet's when importable - ``registry.py`` - or the
    stand-alone ``nn.Module`` below).  The host class provides ``bbox_head``,
    ``with_shared_head`` / ``shared_head`` and, for the sampled head, ``teacher_model``."""

    # ---- StandardRoIReplayHead (:32-50): sampled replay against the teacher -------------
    def init_sampled_replay(self, previous_path, device=None):
        self.replay = False
        self.counter = [0] * 80                                       # :44
        if previous_path is not None and osp.exists(previous_path):
            self.replay = True
            self._sampled = SampledRoIReplay.load(previous_path, device=device)
            (self.bbox_featss, self.cls_targets, self.cls_weights, self.bbox_targets,
             self.bbox_weights, self.roiss) = (getattr(self._sampled, f)
                                               for f in SampledRoIReplay.FIELDS)

    def sampled_replay_losses(self) -> dict:
        """:55-69 - draw 64 stored RoIs, student vs teacher class scores (MSE)."""
        feats, cls_t, cls_w, bbox_t, bbox_w, rois = self._sampled.sample()
        res = self.teacher_replay_loss(feats, [cls_t, cls_w, bbox_t, bbox_w], rois)
        return res["replay_loss"]

    def teacher_replay_loss(self, bbox_feats, sampling_results=None, rois=None) -> dict:
        """:71-104."""
        if getattr(self, "with_shared_head", False):
            bbox_feats = self.shared_head(bbox_feats)
        cls_score, bbox_pred = self.bbox_head(bbox_feats)
        teacher_cls_score, _ = self.teacher_model.bbox_head(bbox_feats)
        losses = {"replay_loss_cls": F.mse_loss(cls_score, teacher_cls_score)}
        return dict(cls_score=cls_score, bbox_pred=bbox_pred, bbox_feats=bbox_feats,
                    replay_loss=losses)

    # ---- StandardMultiPrototypeReplayHead (:377-501): prototype replay -------------------
    def init_prototype_replay(self, previous_path, task_id, task_split, max_prototype,
                              device=None):
        self.replay = False
        self.task_split = list(task_split)
        self.task_id = task_id
        self.max_proto = max_prototype
        self._proto = MultiPrototypeReplay(max_prototype)
        if previous_path is not None and osp.exists(previous_path):
            assert task_id != 1
            self.replay = True
            dev = torch.device(device) if device is not None else torch.device("cuda")
            (bbox_featss, self.cls_targets, self.cls_weights, self.bbox_targets,
             self.bbox_weights, self.roiss) = torch.load(
                osp.join(previous_path, "rois_etc.pth"), map_location=dev)
            previous_cls = range(self.task_split[0], self.task_split[task_id - 1])
            saved = None
            if osp.exists(osp.join(previous_path, "mask.pth")):
                saved = torch.load(osp.join(previous_path, "mask.pth"), map_location="cpu")
            self._proto.build(bbox_featss, self.cls_targets, previous_cls, saved)
            self.bbox_featss = self._proto.bbox_featss
            self.tmp_label = self._proto.tmp_label
            # like the reference (:451-452) the masks go next to the NEXT task's outputs,
            # whatever ``work_dir`` was passed
            torch.save(self._proto.save_idx,
                       osp.join(get_work_dir(previous_path), "mask.pth"))

    def replay_loss(self, bbox_feats, sampling_results=None, rois=None) -> dict:
        """:468-501 - logits of classes < task_split[task_id] plus background;
        cross-entropy on the softmax output (double softmax kept on purpose)."""
        if getattr(self, "with_shared_head", False):                  # :488-489
            bbox_feats = self.shared_head(bbox_feats)
        cls_score, bbox_pred = self.bbox_head(bbox_feats)
        pre_idx = self.task_split[self.task_id]
        kept = torch.cat([cls_score[:, :pre_idx], cls_score[:, -1:]], dim=-1)
        losses = {"replay_loss_cls": F.cross_entropy(kept.softmax(dim=-1),
                                                     self.tmp_label.to(kept.device))}
        return dict(cls_score=cls_score, bbox_pred=bbox_pred, bbox_feats=bbox_feats,
                    replay_loss=losses)

    def prototype_replay_losses(self) -> dict:
        """:458-466 - every prototype, every step, gathered on the device."""
        return self.replay_loss(self._proto.staged())["replay_loss"]


class StandardRoIReplayHead(ReplayHeadMixin, nn.Module):
    """Stand-alone form of the sampled-replay head (:32-69): ``bbox_head`` maps
    (P,12544)-features to ``(cls_score, bbox_pred)``; ``teacher_model`` is attached by the
    runner (nsrunner_roi_replay.py:533)."""

    def __init__(self, bbox_head: nn.Module = None, previous_path=None, device=None, **kwargs):
        super().__init__()
        self.bbox_head = bbox_head
        self.with_shared_head = False
        self.init_sampled_replay(previous_path, device)

    def loss(self, x=None, rpn_results_list=None, batch_data_samples=None, replay=True,
             base_losses=None):
        losses = dict(base_losses or {})
        if self.replay and replay:
            losses.update(self.sampled_replay_losses())
        return losses


class StandardMultiPrototypeReplayHead(ReplayHeadMixin, nn.Module):
    """Constructor keywords and attributes of the reference head (:377-390):
    ``previous_path, task_id, task_split, max_prototype, work_dir``; attributes
    ``replay``, ``bbox_featss``, ``tmp_label``; ``loss`` adds ``replay_loss_cls``.

    Stand-alone form: ``bbox_head`` is any module mapping (P,12544)-features to
    ``(cls_score, bbox_pred)``.  When mmdet is importable ``registry.py`` binds the same
    mixin onto the reference's ``StandardRoIReplayHead``.
    """

    def __init__(self, bbox_head: nn.Module = None, previous_path=None, task_id=1,
                 task_split=(0, 10, 20), max_prototype=10, work_dir=None, device=None,
                 **kwargs):
        super().__init__()
        self.bbox_head = bbox_head
        self.with_shared_head = False
        self.counter = [0] * 80
        self.init_prototype_replay(previous_path, task_id, task_split, max_prototype, device)

    def loss(self, x=None, rpn_results_list=None, batch_data_samples=None, base_losses=None):
        """:454-466.  ``base_losses`` stands for ``super().loss(..., replay=False)``."""
        losses = dict(base_losses or {})
        if self.replay:
            losses.update(self.prototype_replay_losses())
        return losses
