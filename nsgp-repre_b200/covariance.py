"""Per-layer input covariance for NSGP - drop-in for the covariance part of
``BRNullSpaceRunner`` (mmdet/engine/runner/nsrunner_roi_replay.py).

Mirrored surface (same names, argument meaning and error behaviour):

* ``compute_cov(module, fea_in, fea_out)`` - forward hook (:876-916)
* ``update_cov(fea_in, k)``                - rows (N,d) -> running X^T X (:923-934)
* ``fea_in``                               - dict "<module path>.weight" -> (d,d)
* ``cal_fea_in`` tail                      - all-reduce over ranks (:746-749), merge
  with the previous task's covariance.pth (:750-753), ``torch.save`` (:757)

What changed underneath: the hook makes ONE C-ABI call per layer that fuses the
batch mean (:908), the im2col (never materialised), X^T X (:930) and the running
add (:931-934) into the layer's persistent fp32 accumulator in HBM.  The
accumulator lives in an internal (tap-major, upper block-triangular) layout;
``fea_in`` expands it to the reference layout on access.
"""
from __future__ import annotations

import re
from collections import OrderedDict

import ctypes

import torch
import torch.nn as nn

from . import _lib
from ._lib import lib, check, ptr, CovLayout, CovJob, Group, StageGroup


class _LayerAcc:
    __slots__ = ("layout", "acc", "calls", "in_arena")

    def __init__(self, layout, acc, in_arena=False):
        self.layout = layout
        self.acc = acc
        self.calls = 0
        self.in_arena = in_arena


class _JobSet:
    """One forward's worth of staged layers for the grouped launch."""

    def __init__(self):
        self.jobs = []          # [key, geometry, workspace, layer accumulator, alias-of index]
        self.seen = {}          # this forward: (input identity, geometry) -> job index
        self.keep = []          # this forward: staged input tensors
        self.pos = 0
        self.sig = None
        self.table = None
        self.group = None
        self.done = None        # event: the grouped launch has finished reading the set
        self.xs = []            # deferred mode: input tensor of job i (None for an alias)
        self.versions = []      # ... and its version counter when the hook saw it
        self.stage_sig = None   # (unique job indices, B) the staging table was built for
        self.stage_table = None
        self.stage_group = None
        self.rev = 0            # bumped whenever the job list changes (tables are rebuilt)
        self.auto_sms = None    # ((rev, B), SMs of the staging half) chosen by _auto_stage_sms
        self.xs_arr = None      # reusable ctypes pointer table of the staging launch
        self.stage_jobs = None  # the CovJob array the staging table was built from
        self.det = False        # deterministic mode the jobs and tables were built in


class CovarianceHooks:
    """Accumulates the un-centred input covariance of every hooked Conv2d/Linear.

    Args:
        model: the detector (unwrapped module); hooks see ``model.named_modules()``.
        ignore_keys: regex prefixes matched with ``re.match`` like :722-726; the
            reference appends ``roi_head.bbox_head.fc_cls|fc_reg|teacher`` (:354).
    """

    DEFAULT_IGNORE = ["roi_head.bbox_head.fc_cls", "roi_head.bbox_head.fc_reg", "teacher"]

    # SMs the HBM-bound staging of forward i gets while the sliding-window contraction of forward
    # i-1 runs on the others (mode="deferred", nsgp_cov_pipeline_launch): an integer, 0 = no
    # partitioning, "auto" = balanced per job set from the measured scaling of the two kernels
    stage_sms = "auto"
    # Model of the two concurrent kernels of the pipelined pass, fitted on B200
    # (profiles/pipeline_r02.txt, TMA-fed staging, B = 2 / 8 / 16 at 800x1344):
    #   staging on S SMs      t = _STAGE_FLOOR[0] + _STAGE_FLOOR[1] * read
    #                             + (_STAGE_READ * read + _STAGE_WRITE * write) / S
    #                         (GB, ms; from ~56 SMs on the phase is HBM-bound at configs[1])
    #   sliding window kernel t = t_alone * 148 / (148 - S) * (1 + _AC_CONTENTION * S)
    _STAGE_FLOOR = (0.15, 0.07)  # ms, ms per GB read
    _STAGE_READ = 4.5            # SM ms per GB read
    _STAGE_WRITE = 15.8          # SM ms per GB written
    _AC_CONTENTION = 0.0019
    # device time (ms) of the caller's own kernels per forward that should find idle SMs
    # inside the pass (the hot path's own: SGDNSCL.step + the RePRE build, 0.45 ms): both
    # kernels are persistent, so the caller's kernels only run on the side that finishes
    # first; a partition that leaves no such window serialises them behind the pass (+0.7 ms
    # measured).  A caller with much more work than fits (a detector's forward / backward)
    # makes the penalty the same for every S, i.e. the plain balance point is chosen.
    main_stream_ms = 0.45

    def __init__(self, model: nn.Module, ignore_keys=(), add_default_ignores=True,
                 mode="deferred"):
        """``mode``
        * ``"deferred"`` (default): a hook call only records its layer input; at the end of
          the forward (``flush``) ONE grouped staging launch (two when a gather layout needs
          the batch mean first) stages all recorded inputs on a staging stream and ONE
          persistent tcgen05 launch contracts them on a side stream - ~3 launches per
          forward instead of ~90 short ones.  The recorded inputs are kept alive until the
          set is reused and must not be modified in place between the hook and the end of
          the forward (checked through the tensors' version counters; mmdet's R50-FPN,
          RPN and RoI heads satisfy this - use ``"grouped"`` for models that do not).
        * ``"grouped"``: every hook call only STAGES its layer (HBM-bound) into
          that layer's own workspace on the caller's stream; at the end of the forward
          (``flush``) the Gram updates of all staged layers run as ONE persistent
          tcgen05 launch on a side stream, overlapping the next forward.  Two workspace
          sets alternate so the next forward never waits for the launch in flight.
        * ``"immediate"``: stage + contract back to back on the caller's stream, one layer
          at a time.  The bring-up SIMT engine has no grouped launch and always runs this
          way.
        Every result access joins the side stream first."""
        self.model = model
        if mode not in ("deferred", "grouped", "immediate"):
            raise ValueError("mode must be 'deferred', 'grouped' or 'immediate'")
        self.mode = mode
        self._sets = [_JobSet(), _JobSet()]
        self._cur = 0
        self._side = None
        self._pending = False
        self.ignore_keys = list(ignore_keys) + (self.DEFAULT_IGNORE if add_default_ignores else [])
        self._names = {}
        self._layers: "OrderedDict[str, _LayerAcc]" = OrderedDict()
        self._workspace = None
        self._handles = []
        self._merged = {}           # key -> dense tensor added at finalize (old tasks)
        self._inflight = None       # deferred mode: the set staged but not yet contracted
        self._geom_cache = {}       # (key, input shape, kernel, stride, padding, device,
                                    #  deterministic) -> layout, layer
        self._arena = None          # ONE flat fp32 buffer holding every planned accumulator
        self._alt = {}              # key -> _LayerAcc of the other layout kind (see _layer)

    # ------------------------------------------------------------------ hooks
    def check_if_ignore(self, n: str) -> bool:
        return any(re.match(k, n) for k in self.ignore_keys)

    def hooked_modules(self):
        """Same selection as :731-732: every module with a ``weight`` attribute
        whose path is not ignored (BatchNorm hooks fire and do nothing)."""
        return [(n, m) for n, m in self.model.named_modules()
                if hasattr(m, "weight") and not self.check_if_ignore(n)]

    def _plan_arena(self):
        """All accumulators of the hooked Conv2d / Linear modules as views of ONE flat fp32
        arena, so that the end-of-accumulation SUM over ranks (:746-749) is a single
        ``ncclAllReduce`` over one buffer.  The accumulator layout of a layer depends only on
        (Cin, kernel, stride, padding), never on the extent of the map it sees, so it can be
        planned before the first forward.  Keys that only appear later (``update_cov`` with a
        foreign key) get their own allocation and join the reduce as extra buffers."""
        if self._arena is not None or self._layers:
            return
        dev = next((p.device for p in self.model.parameters()), None)
        if dev is None or dev.type != "cuda":
            return
        plan, total = [], 0
        for n, m in self.hooked_modules():
            layout = CovLayout()
            if isinstance(m, nn.Conv2d):
                kh, kw = m.kernel_size
                sh, sw = m.stride
                ph, pw = m.padding if not isinstance(m.padding, str) else (0, 0)
                if lib.nsgp_cov_conv2d_layout(m.in_channels, 64, 64, kh, kw, sh, sw, ph, pw,
                                              layout) != 0:
                    continue
            elif isinstance(m, nn.Linear):
                if lib.nsgp_cov_linear_layout(m.in_features, layout) != 0:
                    continue
            else:
                continue
            elems = (layout.acc_bytes // 4 + 63) // 64 * 64         # 256-byte aligned views
            plan.append((n + ".weight", layout, total, layout.acc_bytes // 4))
            total += elems
        if not plan:
            return
        self._arena = torch.zeros(total, dtype=torch.float32, device=dev)
        for key, layout, off, elems in plan:
            self._layers[key] = _LayerAcc(layout, self._arena[off:off + elems], in_arena=True)

    def register(self):
        self._names = {m: n for n, m in self.model.named_modules()}
        self._plan_arena()
        for _, m in self.hooked_modules():
            self._handles.append(m.register_forward_hook(self.compute_cov))
        # end of a forward of the whole model: launch the grouped contraction
        self._handles.append(self.model.register_forward_hook(lambda *a: self.flush()))
        return self

    def remove(self):
        for h in self._handles:
            h.remove()
        self._handles = []

    # ------------------------------------------------------------- side stream
    def _side_stream(self, device):
        if self._side is None or self._side.device != device:
            # high priority: the persistent contraction kernel gets its CTAs placed as soon
            # as blocks of the staging kernels (caller's stream) retire
            self._side = torch.cuda.Stream(device=device, priority=-1)
        return self._side

    # ------------------------------------------------------------ grouped mode
    def _stage_job(self, x, key, geom, B, layout, la, det):
        js = self._sets[self._cur]
        dev = x.device
        main = torch.cuda.current_stream(dev)
        deferred = self.mode == "deferred"
        if js.pos == 0:
            if js.done is not None:
                main.wait_event(js.done)      # the set's previous launch must be finished
            js.keep.clear()                   # ... and only then may its inputs be recycled
            js.xs = []
            js.versions = []
            if js.det != det:
                # workspaces and tables of the other deterministic mode: rebuild them all
                del js.jobs[:]
                js.sig = None
                js.rev += 1
                js.det = det
        # the same tensor with the same geometry earlier in this forward (e.g. the stage
        # output that feeds both layerN.0.conv1 and the FPN lateral conv): stage it once
        ident = (x.data_ptr(), x._version, tuple(x.shape), geom, B)
        src = js.seen.get(ident)
        pos = js.pos
        st = js.jobs[pos] if pos < len(js.jobs) else None
        if st is not None and st[0] == key and st[1] == geom and st[2].device == dev and \
                st[3] is la and st[4] == src:
            ws = st[2]
        else:
            del js.jobs[pos:]
            ws = js.jobs[src][2] if src is not None else \
                torch.empty(int(layout.workspace_bytes), dtype=torch.uint8, device=dev)
            js.jobs.append([key, geom, ws, la, src])
            js.sig = None
            js.rev += 1
        if src is None:
            if not deferred:
                check(lib.nsgp_cov_conv2d_stage(ptr(x), B, *geom, ptr(ws), ws.numel(),
                                                main.cuda_stream), "nsgp_cov_conv2d_stage")
            js.seen[ident] = pos
            js.keep.append(x)                 # keeps the storage (and its address) alive
        js.xs.append(x if src is None else None)
        js.versions.append((x._version, B))
        js.pos += 1
        la.calls += 1

    def flush(self):
        """Launch the device work of every layer recorded / staged since the last flush
        (called automatically after each forward of the hooked model and by ``join``)."""
        js = self._sets[self._cur]
        if js.pos == 0:
            return
        if len(js.jobs) != js.pos:
            del js.jobs[js.pos:]
            js.sig = None
            js.rev += 1
        js.seen.clear()
        # the tables of this set are built in the mode its forward was recorded in
        lib.nsgp_set_deterministic(1 if js.det else 0)
        dev = js.jobs[0][2].device
        main = torch.cuda.current_stream(dev)
        side = self._side_stream(dev)
        staged = torch.cuda.Event()
        staged.record(main)
        side.wait_event(staged)               # the inputs exist / are staged
        if self.mode == "deferred":
            try:
                self._flush_deferred(js, side)
            except Exception:
                # drop the recorded forward so that the hooks stay usable after the error
                js.pos = 0
                js.keep.clear()
                js.xs, js.versions = [], []
                raise
        else:
            js.keep.clear()
            self._build_group(js, side)
            check(lib.nsgp_group_launch(ptr(js.table), ctypes.byref(js.group), side.cuda_stream),
                  "nsgp_group_launch")
        js.done = torch.cuda.Event()
        js.done.record(side)
        js.pos = 0
        self._cur ^= 1
        self._pending = True

    def _build_group(self, js, stream):
        """(Re)build the contraction table of a job set when its job list changed."""
        if js.sig is not None:
            return
        n = len(js.jobs)
        arr = (CovJob * n)()
        for i, (key, geom, ws, la, _alias) in enumerate(js.jobs):
            j = arr[i]
            (j.Cin, j.H, j.W, j.kh, j.kw, j.sh, j.sw, j.ph, j.pw) = geom
            j.acc, j.workspace, j.workspace_bytes = la.acc.data_ptr(), ws.data_ptr(), ws.numel()
        need = int(lib.nsgp_cov_group_bytes(arr, n))
        if need == 0:
            raise _lib.NsgpError("nsgp_cov_group_bytes failed: %s" %
                                 lib.nsgp_last_error().decode("utf-8", "replace"))
        dev = js.jobs[0][2].device
        if js.table is None or js.table.numel() < need or js.table.device != dev:
            js.table = torch.empty(need, dtype=torch.uint8, device=dev)
        js.group = Group()
        check(lib.nsgp_cov_group_build(arr, n, ptr(js.table), js.table.numel(),
                                       ctypes.byref(js.group), stream.cuda_stream),
              "nsgp_cov_group_build")
        js.sig = True

    def _flush_deferred(self, js, side):
        """Deferred mode, pipelined over forwards: this call stages forward i and contracts
        forward i-1 - the HBM-bound staging kernel and the tensor-bound contraction kernels
        run side by side on disjoint sets of SMs (``nsgp_cov_pipeline_launch``); the
        contraction of the last forward is launched by ``join``.  Round 1 ran the two halves
        back to back (they are a third each of the step) because sharing SMs slowed both."""
        uniq = [i for i, x in enumerate(js.xs) if x is not None]
        for i in uniq:
            if js.xs[i]._version != js.versions[i][0]:
                raise _lib.NsgpError(
                    "input of %s was modified in place after its forward hook ran; "
                    "CovarianceHooks(mode='deferred') stages at the end of the forward - "
                    "use mode='grouped' for this model" % js.jobs[i][0])
        self._build_group(js, side)
        prev = self._inflight
        Bs = {js.versions[i][1] for i in uniq}
        ok = len(Bs) == 1 and all(js.xs[i].data_ptr() % 16 == 0 for i in uniq)
        if not ok:
            # ragged batch sizes / unaligned inputs: per-layer staging launches, no pipelining
            self._launch_inflight(side)
            for i in uniq:
                key, geom, ws, la, _ = js.jobs[i]
                check(lib.nsgp_cov_conv2d_stage(ptr(js.xs[i]), js.versions[i][1], *geom, ptr(ws),
                                                ws.numel(), side.cuda_stream),
                      "nsgp_cov_conv2d_stage")
            self._inflight = js
            return
        B = Bs.pop()
        # jobs that read one tensor with different geometries (layerN.0.conv1 and
        # layerN.0.downsample.0 of a ResNet): the library stages a 1x1 stride-2 operand along
        # with the 1x1 stride-1 one.  Part of the table's signature: the promise is checked
        # against the tensors of every forward.
        same = self._same_input_links([js.jobs[i][1] for i in uniq],
                                      [(js.xs[i].data_ptr(), tuple(js.xs[i].shape)) for i in uniq])
        sig = (js.rev, B, same)
        if js.stage_sig != sig:
            n = len(uniq)
            arr = (CovJob * n)()
            for k, i in enumerate(uniq):
                key, geom, ws, la, _ = js.jobs[i]
                j = arr[k]
                (j.Cin, j.H, j.W, j.kh, j.kw, j.sh, j.sw, j.ph, j.pw) = geom
                j.acc, j.workspace, j.workspace_bytes = la.acc.data_ptr(), ws.data_ptr(), ws.numel()
            need = int(lib.nsgp_cov_stage_group_bytes(arr, n, B))
            if need == 0:
                raise _lib.NsgpError("nsgp_cov_stage_group_bytes failed: %s" %
                                     lib.nsgp_last_error().decode("utf-8", "replace"))
            dev = js.jobs[0][2].device
            if js.stage_table is None or js.stage_table.numel() < need or \
                    js.stage_table.device != dev:
                js.stage_table = torch.empty(need, dtype=torch.uint8, device=dev)
            js.stage_group = StageGroup()
            same_arr = (ctypes.c_int * n)(*same)
            check(lib.nsgp_cov_stage_group_build(arr, n, B, same_arr, ptr(js.stage_table),
                                                 js.stage_table.numel(),
                                                 ctypes.byref(js.stage_group),
                                                 side.cuda_stream),
                  "nsgp_cov_stage_group_build")
            js.stage_sig = sig
            js.stage_jobs = arr                   # kept: the per-launch tensor maps need them
            js.xs_arr = (ctypes.c_void_p * n)()
        xs = js.xs_arr
        for k, i in enumerate(uniq):
            xs[k] = js.xs[i].data_ptr()
        have_prev = prev is not None and prev is not js
        if prev is js:                        # the other set was never used: contract first
            self._launch_inflight(side)
        check(lib.nsgp_cov_pipeline_launch(
            ptr(prev.table) if have_prev else None,
            ctypes.byref(prev.group) if have_prev else None,
            ptr(js.stage_table), ctypes.byref(js.stage_group), js.stage_jobs, xs,
            self._auto_stage_sms(js, B) if self.stage_sms == "auto" else int(self.stage_sms),
            side.cuda_stream), "nsgp_cov_pipeline_launch")
        self._inflight = js

    @staticmethod
    def _same_input_links(geoms, idents):
        """``same_input`` of ``nsgp_cov_stage_group_build``: for every staged job the index of
        the 1x1 stride-1 job that reads the same tensor (``idents``: one hashable per job,
        equal for equal tensors), -1 when there is none or the job is that reader itself."""
        source = {}
        for k, (geom, ident) in enumerate(zip(geoms, idents)):
            if tuple(geom[3:]) == (1, 1, 1, 1, 0, 0):
                source.setdefault(ident, k)
        return tuple(-1 if source.get(ident, k) == k else source[ident]
                     for k, ident in enumerate(idents))

    def _auto_stage_sms(self, js, B):
        """Partition of the SMs between the two concurrent kernels of the pipelined pass
        (model: class attributes above); 0 = run them back to back."""
        if js.auto_sms is not None and js.auto_sms[0] == (js.rev, B):
            return js.auto_sms[1]
        read = write = ac_flops = 0.0
        for i, x in enumerate(js.xs):
            key, (Cin, H, W, kh, kw, sh, sw, ph, pw), ws, la, alias = js.jobs[i]
            autocorr = la.layout.kind == 1
            if x is not None:
                read += 4.0 * B * Cin * H * W
                write += (6.6 if autocorr else 2.0) * 4.0 * Cin * H * W
            if autocorr:
                # 13 displacement blocks on / above the diagonal of the channel-tile grid, 12
                # below; the last tile column issues round_up(C mod 128, 16) columns
                t = -(-Cin // 128)
                last = -(-(Cin - (t - 1) * 128) // 16) * 16
                nsum = sum((13 if rb <= cb else 12) * (128 if cb < t - 1 else last)
                           for rb in range(t) for cb in range(t))
                ac_flops += 3 * 2.0 * 128 * nsum * 32 * H * -(-W // 32)
        t_ac = ac_flops / 680e9                          # ms, alone on 148 SMs
        read, write = read / 1e9, write / 1e9
        floor = self._STAGE_FLOOR[0] + self._STAGE_FLOOR[1] * read
        work = self._STAGE_READ * read + self._STAGE_WRITE * write
        m = float(self.main_stream_ms)
        # no partition: back to back, each on the whole GPU (no window for the caller)
        best, best_t = 0, floor + work / 148.0 + t_ac + min(m, 0.7)
        if t_ac > 0 and work > 0:
            for sms in range(24, 124, 4):
                ts = floor + work / sms
                ta = t_ac * 148.0 / (148 - sms) * (1.0 + self._AC_CONTENTION * sms)
                t = max(ts, ta)
                if m > 0:
                    t += min(m, 0.7) * max(0.0, 1.0 - abs(ts - ta) / m)
                if t < best_t:
                    best, best_t = sms, t
        js.auto_sms = ((js.rev, B), best)
        return best

    def _launch_inflight(self, side):
        """Contract the set that is staged but not yet contracted (no staging to pair with)."""
        prev, self._inflight = self._inflight, None
        if prev is not None:
            check(lib.nsgp_cov_pipeline_launch(ptr(prev.table), ctypes.byref(prev.group), None,
                                               None, None, None, 0, side.cuda_stream),
                  "nsgp_cov_pipeline_launch")

    def consumed_event(self):
        """Event that fires when everything launched on the side stream so far has run, i.e.
        when the layer inputs recorded by the forwards flushed up to now have been read
        (``mode="deferred"`` stages at the end of the forward: a caller that recycles an input
        buffer - the image tensor is the stem's input - waits on this).  None before the
        first flush."""
        if self._side is None:
            return None
        ev = torch.cuda.Event()
        ev.record(self._side)
        return ev

    def join(self):
        """Make the current stream wait for every contraction issued on the side stream."""
        self.flush()
        if self._inflight is not None:
            self._launch_inflight(self._side)
        if self._pending and self._side is not None:
            torch.cuda.current_stream(self._side.device).wait_stream(self._side)
            self._pending = False

    def _ws(self, nbytes: int, device) -> torch.Tensor:
        if self._workspace is None or self._workspace.numel() < nbytes or \
                self._workspace.device != device:
            self._workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        return self._workspace

    def _layer(self, key: str, layout: CovLayout, device) -> _LayerAcc:
        la = self._layers.get(key)
        if la is None or la.acc.device != device:
            if la is not None and la.calls:
                raise _lib.NsgpError("covariance of %s moved from %s to %s" %
                                     (key, la.acc.device, device))
            acc = torch.zeros(layout.acc_bytes // 4, dtype=torch.float32, device=device)
            la = _LayerAcc(layout, acc)
            self._layers[key] = la
            self._geom_cache.clear()
        elif la.layout.d != layout.d:
            raise _lib.NsgpError("covariance dimension of %s changed (%d -> %d)" %
                                 (key, la.layout.d, layout.d))
        elif la.layout.kind != layout.kind or la.layout.d_int != layout.d_int:
            # One key hooked at several extents (the RPN convs are shared by the five FPN
            # levels, :893-896): a map smaller than 3 px cannot use the autocorrelation form
            # of a 3x3 conv.  The reference simply adds the Grams; here such a call goes to a
            # second accumulator of the generic layout and the two are summed on read.
            alt = self._alt.get(key)
            if alt is None or alt.acc.device != device:
                alt = _LayerAcc(layout, torch.zeros(layout.acc_bytes // 4, dtype=torch.float32,
                                                    device=device))
                self._alt[key] = alt
            elif alt.layout.kind != layout.kind or alt.layout.d_int != layout.d_int:
                raise _lib.NsgpError("%s: a third accumulator layout (kind %d, %d rows) for one "
                                     "key" % (key, layout.kind, layout.d_int))
            return alt
        return la

    @torch.no_grad()
    def compute_cov(self, module, fea_in, fea_out):
        """Forward hook, same signature and return value (None) as :876-916."""
        if not self._names:
            self._names = {m: n for n, m in self.model.named_modules()}
        name = self._names[module] + ".weight"
        x = fea_in[0]
        if isinstance(module, nn.Linear):
            self._accumulate_linear(x, name)
        elif isinstance(module, nn.Conv2d):
            self._accumulate_conv(x, name, module.kernel_size, module.stride, module.padding)
        return None

    def _accumulate_conv(self, x, key, kernel_size, stride, padding):
        _lib.require_cuda(x, "layer input")
        if x.dim() != 4:
            raise _lib.NsgpError("Conv2d input must be (B,C,H,W)")
        x = x.detach()
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        # layout + accumulator of (key, extent): looked up once, the hook runs per layer per
        # forward on the training thread.  The workspace size depends on the deterministic mode.
        det = _lib.deterministic()
        ck = (key, x.shape, kernel_size, stride, padding, x.device, det)
        hit = self._geom_cache.get(ck)
        if hit is None:
            B, Cin, H, W = x.shape
            kh, kw = kernel_size
            sh, sw = stride
            ph, pw = padding
            layout = CovLayout()
            check(lib.nsgp_cov_conv2d_layout(Cin, H, W, kh, kw, sh, sw, ph, pw, layout),
                  "nsgp_cov_conv2d_layout")
            la = self._layer(key, layout, x.device)
            hit = ((Cin, H, W, kh, kw, sh, sw, ph, pw), B, layout, la)
            self._geom_cache[ck] = hit
        (Cin, H, W, kh, kw, sh, sw, ph, pw), B, layout, la = hit
        # the bring-up engine has no grouped launch
        if self.mode in ("grouped", "deferred") and _lib.engine() == 0:
            self._stage_job(x, key, (Cin, H, W, kh, kw, sh, sw, ph, pw), B, layout, la, det)
            return
        ws = self._ws(layout.workspace_bytes, x.device)
        check(lib.nsgp_cov_conv2d_accumulate(
            ptr(x), B, Cin, H, W, kh, kw, sh, sw, ph, pw, ptr(la.acc), ptr(ws), ws.numel(),
            _lib.current_stream(x.device)), "nsgp_cov_conv2d_accumulate")
        la.calls += 1

    def _accumulate_linear(self, x, key):
        _lib.require_cuda(x, "layer input")
        x = x.detach()
        d = x.shape[-1]
        if x.dim() != 2:
            # torch.mean(x, 0, True) on a (B, ..., d) input keeps the inner dims as rows
            # (:901); the Gram of those rows is the reference result.
            rows = x.float().mean(dim=0).reshape(-1, d)
            return self.update_cov(rows, key)
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        layout = CovLayout()
        check(lib.nsgp_cov_linear_layout(d, layout), "nsgp_cov_linear_layout")
        self.join()                  # same accumulator may have a contraction in flight
        la = self._layer(key, layout, x.device)
        ws = self._ws(layout.workspace_bytes, x.device)
        check(lib.nsgp_cov_linear_accumulate(ptr(x), x.shape[0], d, ptr(la.acc), ptr(ws),
                                             ws.numel(), _lib.current_stream(x.device)),
              "nsgp_cov_linear_accumulate")
        la.calls += 1

    @torch.no_grad()
    def update_cov(self, fea_in: torch.Tensor, k: str):
        """Reference signature (:923): rows X (N,d) -> fea_in[k] (+)= X^T X.
        Routed through the conv entry point as a 1x1 "image" (d, 1, N)."""
        _lib.require_cuda(fea_in, "fea_in")
        xt = fea_in.detach().float().t().contiguous()          # (d, N), K-major
        d, N = xt.shape
        self._accumulate_conv(xt.view(1, d, 1, N), k, (1, 1), (1, 1), (0, 0))

    # ---------------------------------------------------------------- results
    def _finalize(self, key: str) -> torch.Tensor:
        self.join()
        la = self._layers[key]
        d = la.layout.d
        out = torch.empty(d, d, dtype=torch.float32, device=la.acc.device)
        check(lib.nsgp_cov_finalize(ptr(la.acc), la.layout, ptr(out), 0,
                                    _lib.current_stream(out.device)), "nsgp_cov_finalize")
        alt = self._alt.get(key)
        if alt is not None:
            check(lib.nsgp_cov_finalize(ptr(alt.acc), alt.layout, ptr(out), 1,
                                        _lib.current_stream(out.device)), "nsgp_cov_finalize")
        if key in self._merged:
            out += self._merged[key].to(out.device)
        return out

    def _live(self):
        """Keys that received at least one hook call (the reference only creates a key when
        its module fires, :931-934)."""
        return [k for k, la in self._layers.items()
                if la.calls or (k in self._alt and self._alt[k].calls)]

    @property
    def fea_in(self) -> dict:
        """dict "<module path>.weight" -> (d,d) fp32, reference layout (:931-934)."""
        return {k: self._finalize(k) for k in self._live()}

    def keys(self):
        return self._live()

    def reduce_buffers(self):
        """The fp32 buffers the SUM over ranks runs on: the arena first, then every
        accumulator allocated outside it."""
        bufs = [] if self._arena is None else [self._arena]
        bufs += [la.acc for la in self._layers.values() if not la.in_arena]
        bufs += [la.acc for la in self._alt.values()]
        return bufs

    def reset(self):
        self.join()
        for b in self.reduce_buffers():
            b.zero_()
        for la in list(self._layers.values()) + list(self._alt.values()):
            la.calls = 0
        self._merged = {}

    # ------------------------------------------------- cal_fea_in tail (:746-757)
    def all_reduce(self, group=None):
        """SUM over ranks of every accumulator, as ``all_reduce_dict(self.fea_in)``
        (:746-749), in place on the fp32 sums, NCCL over NVLink (gloo in the CPU tests)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or \
                dist.get_world_size(group) == 1 or not self._layers:
            return
        self.join()
        # in place on the flat arena: ONE ncclAllReduce over NVLink for every planned layer;
        # accumulators outside the arena (foreign update_cov keys, second-layout keys) follow
        # as one coalesced group call
        accs = self.reduce_buffers()
        if len(accs) == 1:
            dist.all_reduce(accs[0], op=dist.ReduceOp.SUM, group=group)
            return
        if dist.get_backend(group) == "nccl":
            try:
                from torch.distributed.distributed_c10d import _coalescing_manager
                with _coalescing_manager(group=group, device=accs[0].device, async_ops=True) as cm:
                    for a in accs:
                        dist.all_reduce(a, op=dist.ReduceOp.SUM, group=group)
                cm.wait()
                return
            except (ImportError, TypeError):
                pass
        works = [dist.all_reduce(a, op=dist.ReduceOp.SUM, group=group, async_op=True) for a in accs]
        for w in works:
            w.wait()

    def merge_previous(self, old_fea_in: dict):
        """``fea_in[k] + old_fea_in[k]`` for task_id != 1 (:750-753); keys of the
        current run that are ignored are dropped there, missing old keys raise
        KeyError like the reference's dict lookup."""
        for k in self._live():
            self._merged[k] = old_fea_in[k] if k not in self._merged else \
                self._merged[k] + old_fea_in[k]

    def save(self, path: str):
        """``torch.save(self.fea_in, fea_in_save_path)`` (:757), same pickle format."""
        torch.save(self.fea_in, path)

    @torch.no_grad()
    def cal_fea_in(self, batches, forward=None, save_path=None, previous=None, group=None):
        """The accumulation loop + tail of ``cal_fea_in`` (:731-763) on an iterable
        of already pre-processed input batches.  ``forward(model, batch)``
        defaults to ``model(batch)`` (the reference calls
        ``model(inputs, data_samples, mode='nullspace')``)."""
        self.register()
        was_training = self.model.training
        self.model.eval()
        try:
            for batch in batches:
                (forward or (lambda m, b: m(b)))(self.model, batch)
        finally:
            self.remove()
            self.model.train(was_training)
        self.all_reduce(group)
        if previous is not None:
            self.merge_previous(previous)
        out = self.fea_in
        if save_path is not None:
            torch.save(out, save_path)
        return out


BRNullSpaceCovariance = CovarianceHooks
