"""ctypes binding of ``lib/libnsgp_repre_b200.so`` (C ABI: include/nsgp_repre_b200.h)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libnsgp_repre_b200.so")
# developers only: the -DNSGP_BRINGUP build (make BRINGUP=1) with the SIMT cross-check engine
if os.environ.get("NSGP_BRINGUP_LIB") == "1":
    LIB_PATH = os.path.join(_HERE, "lib", "libnsgp_repre_b200_bringup.so")

if not os.path.isfile(LIB_PATH):
    raise ImportError(
        "nsgp_repre_b200: %s is missing - build it with "
        "`make -C nsgp-repre_b200/csrc` (or __graft_entry__.build()). "
        "There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

c_void_p, c_int, c_size_t, c_float, c_double = C.c_void_p, C.c_int, C.c_size_t, C.c_float, C.c_double


class CovLayout(C.Structure):
    _fields_ = [("d", c_int), ("d_int", c_int), ("taps", c_int), ("ld", c_int), ("kind", c_int),
                ("acc_bytes", c_size_t), ("workspace_bytes", c_size_t)]


class SgdTensor(C.Structure):
    _fields_ = [("w", c_void_p), ("g", c_void_p), ("buf", c_void_p),
                ("numel", C.c_longlong), ("first_step", c_int), ("layer", c_int)]


class ProjLayer(C.Structure):
    _fields_ = [("cout", c_int), ("d", c_int), ("pt_hi", c_void_p), ("pt_lo", c_void_p),
                ("u_hi", c_void_p), ("u_lo", c_void_p), ("r", c_int), ("scale", c_float),
                ("ut_hi", c_void_p), ("ut_lo", c_void_p), ("un_hi", c_void_p),
                ("un_lo", c_void_p), ("t", c_void_p), ("t_hi", c_void_p), ("t_lo", c_void_p)]


class Group(C.Structure):
    _fields_ = [("kind", c_int), ("n_problems", c_int * 4), ("n_items", c_int * 4),
                ("off_probs", c_size_t * 4), ("off_items", c_size_t * 4), ("bytes", c_size_t)]


class SgdPlan(C.Structure):
    _fields_ = [("n_tensors", c_int), ("total_chunks", c_int), ("all_have_buf", c_int),
                ("off_chunks", c_size_t), ("off_group", c_size_t), ("off_group2", c_size_t),
                ("group", Group), ("group2", Group), ("t_arena", c_void_p),
                ("t_elems", c_size_t), ("bytes", c_size_t)]


class StageGroup(C.Structure):
    _fields_ = [("n_jobs", c_int), ("B", c_int), ("n_items", c_int * 2), ("off_jobs", c_size_t),
                ("off_items", c_size_t * 2), ("off_xs", c_size_t), ("bytes", c_size_t),
                ("n_items_tma", c_int), ("pad", c_int), ("off_items_tma", c_size_t),
                ("off_maps", c_size_t)]


class EwcTensor(C.Structure):
    _fields_ = [("p", c_void_p), ("importance", c_void_p), ("old_params", c_void_p),
                ("grad", c_void_p), ("numel", C.c_longlong), ("tasks", c_int)]


class CovJob(C.Structure):
    _fields_ = [("Cin", c_int), ("H", c_int), ("W", c_int), ("kh", c_int), ("kw", c_int),
                ("sh", c_int), ("sw", c_int), ("ph", c_int), ("pw", c_int),
                ("acc", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t)]


# name -> (restype, argtypes); every symbol of include/nsgp_repre_b200.h
SIGNATURES = {
    "nsgp_abi_version": (c_int, []),
    "nsgp_last_error": (C.c_char_p, []),
    "nsgp_launch_count": (C.c_ulonglong, []),
    "nsgp_set_deterministic": (c_int, [c_int]),
    "nsgp_get_deterministic": (c_int, []),
    "nsgp_profile_enable": (c_int, [c_int]),
    "nsgp_profile_read": (c_int, [c_int, C.POINTER(c_double), C.POINTER(C.c_ulonglong)]),
    "nsgp_cov_conv2d_layout": (c_int, [c_int] * 9 + [C.POINTER(CovLayout)]),
    "nsgp_cov_linear_layout": (c_int, [c_int, C.POINTER(CovLayout)]),
    "nsgp_cov_conv2d_accumulate": (c_int, [c_void_p] + [c_int] * 10 +
                                   [c_void_p, c_void_p, c_size_t, c_void_p]),
    "nsgp_cov_conv2d_stage": (c_int, [c_void_p] + [c_int] * 10 + [c_void_p, c_size_t, c_void_p]),
    "nsgp_cov_conv2d_contract": (c_int, [c_int] * 9 + [c_void_p, c_void_p, c_size_t, c_void_p]),
    "nsgp_cov_linear_accumulate": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p,
                                           c_size_t, c_void_p]),
    "nsgp_cov_finalize": (c_int, [c_void_p, C.POINTER(CovLayout), c_void_p, c_int, c_void_p]),
    "nsgp_projector_prepare": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "nsgp_sgd_step_workspace_bytes": (c_size_t, [c_int, c_int]),
    "nsgp_sgd_nscl_step": (c_int, [C.POINTER(SgdTensor), c_int, C.POINTER(ProjLayer), c_int,
                                   c_double, c_double, c_double, c_double, c_int,
                                   c_void_p, c_size_t, c_void_p]),
    "nsgp_sgd_plan_bytes": (c_size_t, [C.POINTER(SgdTensor), c_int, C.POINTER(ProjLayer), c_int]),
    "nsgp_sgd_plan_build": (c_int, [C.POINTER(SgdTensor), c_int, C.POINTER(ProjLayer), c_int,
                                    c_void_p, c_size_t, c_void_p, c_size_t, C.POINTER(SgdPlan),
                                    c_void_p]),
    "nsgp_projector_prepare_lowrank": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p,
                                               c_void_p, c_void_p, c_void_p]),
    "nsgp_sgd_plan_step": (c_int, [C.POINTER(SgdTensor), c_int, C.POINTER(ProjLayer), c_int,
                                   c_void_p, C.POINTER(SgdPlan), c_double, c_double, c_double,
                                   c_double, c_int, c_void_p]),
    "nsgp_cov_group_bytes": (c_size_t, [C.POINTER(CovJob), c_int]),
    "nsgp_cov_group_build": (c_int, [C.POINTER(CovJob), c_int, c_void_p, c_size_t,
                                     C.POINTER(Group), c_void_p]),
    "nsgp_cov_stage_group_bytes": (c_size_t, [C.POINTER(CovJob), c_int, c_int]),
    "nsgp_cov_stage_group_build": (c_int, [C.POINTER(CovJob), c_int, c_int, C.POINTER(c_int),
                                           c_void_p, c_size_t,
                                           C.POINTER(StageGroup), c_void_p]),
    "nsgp_cov_stage_group_launch": (c_int, [c_void_p, C.POINTER(StageGroup), C.POINTER(CovJob),
                                            C.POINTER(c_void_p), c_void_p]),
    "nsgp_group_launch": (c_int, [c_void_p, C.POINTER(Group), c_void_p]),
    "nsgp_cov_pipeline_launch": (c_int, [c_void_p, C.POINTER(Group), c_void_p,
                                         C.POINTER(StageGroup), C.POINTER(CovJob),
                                         C.POINTER(c_void_p), c_int, c_void_p]),
    "repre_class_index": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                  c_void_p]),
    "repre_segment_mean": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int,
                                   c_void_p, c_void_p]),
    "repre_segment_var": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int,
                                  c_void_p, c_void_p, c_void_p]),
    "repre_cosine_count_workspace_bytes": (c_size_t, [c_int, c_int]),
    "repre_cosine_count": (c_int, [c_void_p, c_int, c_void_p, c_int, c_float, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "repre_cosine_count_batched_workspace_bytes": (c_size_t, [C.POINTER(C.c_int32), c_int, c_int]),
    "repre_cosine_count_batched": (c_int, [c_void_p, c_int, c_void_p, C.POINTER(C.c_int32), c_int,
                                           c_float, c_void_p, c_void_p, c_void_p, c_size_t,
                                           c_void_p]),
    "repre_greedy_segments_workspace_bytes": (c_size_t, [C.POINTER(C.c_int32), c_int, c_int]),
    "repre_greedy_segments": (c_int, [c_void_p, c_void_p, c_void_p, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32), c_int, c_int, c_void_p,
                                      C.POINTER(C.c_int32), c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_size_t, c_void_p]),
    "repre_build_prototypes_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "repre_build_prototypes": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                       c_float, c_int, c_void_p, C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int32), c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_size_t, c_int, c_void_p]),
    "repre_segment_mean_dev": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                       c_int, c_void_p, c_void_p]),
    "repre_replay_gather": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int,
                                    C.c_uint64, c_void_p, c_void_p]),
    "repre_replay_gather_rois": (c_int, [c_void_p] * 7 + [c_int, c_int] + [c_void_p] * 7),
    "repre_kmeans_assign_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "repre_kmeans_assign": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p,
                                    c_void_p, c_size_t, c_void_p]),
    "repre_roi_align": (c_int, [C.POINTER(c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(c_float), c_int, c_int, c_int, c_void_p, c_int, c_int,
                                c_int, c_int, c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "repre_roi_align_backward": (c_int, [C.POINTER(c_void_p), C.POINTER(C.c_int32),
                                         C.POINTER(C.c_int32), C.POINTER(c_float), c_int, c_int,
                                         c_int, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                         c_void_p, c_void_p, c_void_p]),
    "nsgp_ewc_table_bytes": (c_size_t, [c_int]),
    "nsgp_ewc_accumulate": (c_int, [C.POINTER(EwcTensor), c_int, c_float, c_float, c_void_p,
                                    c_size_t, c_void_p]),
    "nsgp_ewc_penalty": (c_int, [C.POINTER(EwcTensor), c_int, c_float, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    "nsgp_ewc_penalty_backward": (c_int, [C.POINTER(EwcTensor), c_int, c_float, c_void_p,
                                          c_void_p, c_size_t, c_void_p]),
    "nsgp_pseudo_label_merge": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_int, c_float, c_float, c_double, c_void_p, c_void_p,
                                        c_void_p, c_void_p]),
    "nsgp_split_tf32": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "nsgp_gemm_nt": (c_int, [c_void_p] * 4 + [c_int] * 3 + [c_void_p, c_int, c_void_p]),
}

# symbols of the bring-up build only (include/nsgp_repre_b200.h, #ifdef NSGP_BRINGUP)
BRINGUP_SIGNATURES = {
    "nsgp_set_engine": (c_int, [c_int]),
    "nsgp_get_engine": (c_int, []),
    "nsgp_debug_read_counters": (c_int, [C.POINTER(C.c_ulonglong), c_int]),
    "nsgp_debug_mma_rate": (c_int, [c_int, c_int, c_void_p, c_int, c_void_p]),
    "nsgp_debug_tma_probe": (c_int, [c_void_p, C.c_longlong, c_int, c_int, c_int, c_int, c_void_p,
                                     c_int, c_void_p]),
    "nsgp_debug_tma3d_probe": (c_int, [c_void_p, C.c_longlong, c_int, c_int, c_int, c_int, c_void_p,
                                       c_int, c_void_p]),
    "nsgp_debug_bulk_probe": (c_int, [c_void_p, C.c_longlong, c_int, c_int, c_void_p, c_int,
                                      c_void_p]),
    "nsgp_debug_timeline_read": (c_int, [C.POINTER(C.c_ulonglong), C.POINTER(c_int), c_int]),
    "nsgp_debug_occupy": (c_int, [c_int, c_size_t, C.c_longlong, c_int, c_void_p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here = ABI mismatch, fail loudly
    _fn.restype = _res
    _fn.argtypes = _args

HAS_BRINGUP = hasattr(lib, "nsgp_set_engine")
if HAS_BRINGUP:
    for _name, (_res, _args) in BRINGUP_SIGNATURES.items():
        _fn = getattr(lib, _name)
        _fn.restype = _res
        _fn.argtypes = _args


def engine() -> int:
    """0 = tcgen05 (the only engine of the shipped library)."""
    return int(lib.nsgp_get_engine()) if HAS_BRINGUP else 0

if lib.nsgp_abi_version() != 1:
    raise ImportError("nsgp_repre_b200: ABI version mismatch")


class NsgpError(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib.nsgp_last_error().decode("utf-8", "replace")
        raise NsgpError("%s failed (rc=%d): %s" % (what, rc, msg))


def ptr(t) -> int:
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream(device=None) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t, name="tensor"):
    if not t.is_cuda:
        raise NsgpError("%s must live on a CUDA device (there is no CPU fallback)" % name)


def deterministic() -> bool:
    """Mirror ``torch.are_deterministic_algorithms_enabled()`` into the library (size queries and
    table builds read it) and return it.  Called before every build or one-shot call; every cache
    of a table, layout or plan has the returned mode in its key, so switching rebuilds."""
    import torch
    on = bool(torch.are_deterministic_algorithms_enabled())
    lib.nsgp_set_deterministic(1 if on else 0)
    return on


def alert_not_deterministic(name: str) -> None:
    """torch's contract for an operation without a deterministic implementation: raise
    RuntimeError under ``torch.use_deterministic_algorithms(True)``, warn under
    ``warn_only=True``, nothing when the switch is off."""
    import torch
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = ("%s does not have a deterministic implementation, but you set "
           "'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this "
           "operation, or you can use the 'warn_only=True' option, if that's acceptable for your "
           "application." % name)
    if torch.is_deterministic_algorithms_warn_only_enabled():
        import warnings
        warnings.warn(msg, UserWarning, stacklevel=3)
    else:
        raise RuntimeError(msg)


PROFILE_KINDS = {"gram": 0, "gemm": 1, "stage": 2, "sgd": 3, "repre": 4}


PROFILE_ON = False


def profile_enable(on: bool) -> None:
    global PROFILE_ON
    PROFILE_ON = bool(on)
    lib.nsgp_profile_enable(1 if on else 0)


def profile_read() -> dict:
    """{kind: (milliseconds, launches)} accumulated since the last read."""
    out = {}
    for name, k in PROFILE_KINDS.items():
        ms, n = c_double(0.0), C.c_ulonglong(0)
        check(lib.nsgp_profile_read(k, C.byref(ms), C.byref(n)), "nsgp_profile_read")
        out[name] = (ms.value, int(n.value))
    return out


def launch_count() -> int:
    return int(lib.nsgp_launch_count())
