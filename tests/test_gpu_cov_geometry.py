"""The covariance pass at every layout, staging routine, channel count and map edge, element by
element against the oracle's unfold + mm evaluated in fp64 on the device.

The full-size tests check a few R50-FPN geometries by relative Frobenius norm.  A missing edge-row,
edge-column or corner correction of the sliding-window layout moves an element by about 1/(H*W) of
its size, which no such bar sees at full extents.  Here the maps are small, their border rows,
columns and corners are several times larger than the interior, every channel has its own scale,
and every element (i, j) must satisfy

    |got - want| <= TAU * sqrt(want_ii * want_jj)

By Cauchy-Schwarz that is the scale of the error of a 3xTF32 dot product of columns i and j, so
the bar is as strict for a small edge term as for the diagonal.  TAU is the bar of the full-size
tests (DESIGN.md section 4: accumulation bias <= ~1.1e-5).

``test_every_staging_route_is_reached`` (no GPU) restates the routine choice of the staging
planner and asserts that the grid below reaches every routine it can pick.
"""
import math
import os
import zlib

import pytest
import torch
import torch.nn as nn

from conftest import rel_fro
from oracle import restated as O

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

TAU = 3e-5
FRO = 2e-5
ASYM = 1e-6

KERNEL = {"autocorr": "autocorrelation", "flat": "flat", "implicit": "implicit",
          "explicit": "explicit", "linear": "linear"}


# ------------------------------------------------------------------------------------ the grid
def _g(C, H, W, k, s=(1, 1), p=(1, 1), Bs=(1, 2), det=False):
    kh, kw = (k, k) if isinstance(k, int) else k
    sh, sw = (s, s) if isinstance(s, int) else s
    ph, pw = (p, p) if isinstance(p, int) else p
    return (C, H, W, kh, kw, sh, sw, ph, pw), tuple(Bs), det


GRID = [
    # ---- 3x3 s1 p1, autocorrelation layout: channels 8 ... 264, maps around the 48-row x
    #      32-column work items of the sliding-window kernel, both staging routines
    _g(8, 3, 3, 3),                          # every pixel an edge or corner; batch mean + scalar
    _g(16, 4, 4, 3, Bs=(1, 3)),              # img % 256 = 0, W % 4 = 0: TMA route, run-time B
    _g(8, 97, 65, 3, det=True),              # rows past two items, columns past two strips
    _g(16, 48, 33, 3, Bs=(1, 2, 16), det=True),  # W % 4 != 0, img % 256 = 0: TMA batch mean; B = 16
    _g(120, 47, 31, 3, Bs=(1, 8), det=True),  # 120 channels: last block issues 128 columns
    _g(128, 48, 32, 3, Bs=(1, 8), det=True),  # exactly one work item and one channel block
    _g(136, 49, 33, 3, det=True),            # partial last block of 8 channels; 48 + 1 rows
    _g(136, 4, 32, 3, Bs=(1, 3), det=True),  # partial block on the TMA route
    _g(200, 97, 36, 3, Bs=(1, 16), det=True),  # last block 72 channels; register route
    _g(200, 49, 32, 3, det=True),            # partial block, TMA route
    _g(264, 3, 4, 3, Bs=(1, 8), det=True),   # two full blocks + 8; three rows
    _g(264, 47, 65, 3, Bs=(1, 3), det=True),  # largest d of the grid (2376); batch mean
    _g(264, 48, 36, 3, det=True),            # TMA route, two blocks + 8
    _g(16, 97, 3, 3),                        # narrowest autocorrelation map
    _g(128, 3, 65, 3),                       # shallowest
    _g(120, 4, 36, 3),                       # W % 4 = 0, img % 256 != 0: register route
    _g(8, 47, 4, 3, Bs=(1, 16)),
    _g(8, 48, 31, 3),
    _g(16, 49, 31, 3, Bs=(2,)),
    _g(136, 97, 32, 3, Bs=(2,), det=True),
    _g(8, 3, 33, 3, Bs=(1, 3)),
    # ---- 3x3 s1 p1 off the autocorrelation layout (implicit)
    _g(16, 2, 8, 3),                         # H < 3, W % 4 = 0: kSt3x3Vec
    _g(16, 1, 4, 3, Bs=(1, 3)),              # one row, kSt3x3Vec
    _g(16, 2, 5, 3),                         # H < 3, W % 4 != 0: gather
    _g(16, 6, 2, 3),                         # W < 3
    _g(8, 1, 1, 3),                          # 1 x 1 map: eight of nine taps read padding only
    _g(24, 2, 2, 3, Bs=(1, 16)),
    # ---- stride 2
    _g(64, 9, 16, 3, s=2),                   # odd H, img % 256 = 0: kStS2x3
    _g(32, 16, 8, 3, s=2, Bs=(1, 8)),        # even H, kStS2x3
    _g(16, 17, 32, 3, s=2, Bs=(1, 16)),      # odd H, kStS2x3 with 3-row boxes
    _g(24, 9, 12, 3, s=2),                   # W % 4 = 0, img % 256 != 0: gather; 8-row boxes
    _g(40, 10, 13, 3, s=2, Bs=(1, 3), det=True),  # W % 4 != 0; 40 rows per tap: 8-row boxes
    _g(136, 7, 9, 3, s=2, det=True),         # 136 rows per tap: 8-row boxes, tiles span taps
    _g(16, 11, 12, 3, s=2, p=0),             # 3x3 s2 p0
    _g(16, 9, 7, 1, s=2, p=0),               # 1x1 s2 at odd W: strided gather, no batch mean
    _g(16, 8, 8, 1, s=2, p=0, Bs=(1, 8)),
    # ---- implicit layout, other kernels / strides / paddings
    _g(16, 7, 9, (1, 3), p=(0, 1)),
    _g(24, 8, 6, (3, 1), p=(1, 0), Bs=(1, 3)),
    _g(8, 5, 20, (1, 7), p=(0, 3)),
    _g(16, 12, 5, (5, 1), p=(2, 0)),
    _g(16, 12, 5, (5, 1), p=0),
    _g(16, 10, 12, 2, s=2, p=0, Bs=(1, 8)),
    _g(8, 13, 14, 3, s=3),                   # three row phases
    _g(16, 9, 12, 3, s=(1, 2)),
    _g(16, 8, 8, 3, p=0),
    _g(16, 6, 7, 3, p=2),
    _g(16, 5, 6, 1, p=1),                    # 1x1 with padding is not the flat layout
    _g(24, 9, 11, (1, 3), p=(0, 1)),         # multi-tap Grams with 8-row boxes
    _g(40, 6, 10, (1, 3), p=(0, 1)),
    _g(136, 5, 8, (1, 3), p=(0, 1), det=True),
    _g(16, 16, 16, (1, 3), p=(0, 1), Bs=(2,)),  # img % 256 = 0: TMA batch mean + gather
    # ---- flat 1x1
    _g(64, 8, 8, 1, p=0),                    # H*W % 4 = 0, TMA route
    _g(16, 7, 9, 1, p=0, Bs=(1, 3)),         # H*W % 4 != 0: batch mean + gather
    _g(24, 6, 10, 1, p=0),                   # register route
    _g(136, 9, 12, 1, p=0),
    _g(8, 23, 89, 1, p=0, det=True),         # K = 2047: one K chain is 64 blocks of 32
    _g(8, 32, 64, 1, p=0, det=True),         # K = 2048
    _g(8, 3, 683, 1, p=0, det=True),         # K = 2049
    _g(16, 63, 65, 1, p=0, det=True),        # K = 4095
    _g(16, 64, 64, 1, p=0, Bs=(1, 8), det=True),  # K = 4096
    _g(16, 17, 241, 1, p=0, det=True),       # K = 4097
    # ---- explicit layout (Cin % 8 != 0, or more than 9 taps)
    _g(3, 9, 11, 3),                         # odd C*H*W: unaligned images, no batch mean
    _g(3, 16, 16, 3),                        # img % 256 = 0: TMA batch mean, Wout % 4 = 0
    _g(12, 8, 8, 1, p=0),                    # d = 12
    _g(20, 9, 12, 5, p=2, det=True),         # d = 500, Wout % 4 = 0
    _g(12, 7, 9, 3, Bs=(1, 3)),              # batch mean, Wout % 4 != 0
    _g(15, 6, 8, 3),                         # d = 135, just above 128
    _g(29, 6, 7, 3, det=True),               # d = 261, just above 256
    _g(3, 9, 15, 3, s=2),                    # odd image, Wout = 8: row-aligned items, B > 1
    _g(3, 16, 48, 5, p=1, det=True),         # TMA batch mean, Wout = 46
    _g(3, 32, 40, 7, s=2, p=3, det=True),    # the stem's kernel
    _g(8, 9, 10, 5, p=2, det=True),          # Cin % 8 = 0 but 25 taps
    _g(20, 5, 5, 1, p=0),
]

# the sliding-window layer in every forward of the grid: the pipelined pass contracts its
# previous forward next to the staging of the layer under test
COMPANION = (16, 8, 16, 3, 3, 1, 1, 1, 1)

MODES = [("deferred", "auto"), ("deferred", 40), ("grouped", "auto"), ("immediate", "auto")]


def _gid(geom):
    C, H, W, kh, kw, sh, sw, ph, pw = geom
    return "c%d_%dx%d_k%dx%d_s%dx%d_p%dx%d" % (C, H, W, kh, kw, sh, sw, ph, pw)


def _cases():
    out = []
    for geom, Bs, _det in GRID:
        for B in Bs:
            for mode, sms in MODES:
                out.append(pytest.param(geom, B, mode, sms,
                                        id="%s_b%d_%s-%s" % (_gid(geom), B, mode, sms)))
    return out


# ---------------------------------------------------- restated layout and routine choice
# Mirrors make_conv_geom (geometry.h: the layout) and plan_stage_job (stage.cu: the routines that
# stage a layer, for deferred mode's staging table and for the per-layer launches of grouped and
# immediate modes and of deferred mode's fallback).  Change them together.
def _layout(C, H, W, kh, kw, sh, sw, ph, pw):
    if (kh, kw, sh, sw, ph, pw) == (3, 3, 1, 1, 1, 1) and C % 8 == 0 and H >= 3 and W >= 3:
        return "autocorr"
    if (kh, kw, ph, pw) == (1, 1, 0, 0) and C % 8 == 0:
        return "flat"
    return "implicit" if kh * kw <= 9 and C % 8 == 0 else "explicit"


def _tma_enabled(B):
    """stage_tma_enabled: the TMA box of B images fits a ring of at least two stages."""
    if not 1 <= B <= 32:
        return False
    rows = 8 if 8 * B <= 32 else 4 if 4 * B <= 48 else max(48 // B, 1)
    ring = 192 * 1024 + (32 * 1024 if B in (1, 2, 4, 8) else 0)
    return min(ring // (B * rows * 1024), 12) >= 2


def _sub_pair_ok(sub, full, B):
    """stage_sub_pair_ok: a 1x1 s2 job staged along with the 1x1 s1 job on the same tensor."""
    C, H, W = full[:3]
    return (_tma_enabled(B) and C * H * W % 256 == 0 and W % 4 == 0 and
            _layout(*full) == "flat" and _layout(*sub) == "flat" and full[5:7] == (1, 1) and
            sub[5:7] == (2, 2) and sub[:3] == full[:3] and ((W - 1) // 2 + 1) * 2 == W)


def _routine(geom, B, tma, aligned, paired=False):
    """Routines that stage one layer (plan_stage_job).  ``tma``: the TMA kernel may take the layer
    (staging tables); ``aligned``: x % 16 == 0 (staging tables require it)."""
    C, H, W, kh, kw, sh, sw, ph, pw = geom
    mode = _layout(*geom)
    img = C * H * W
    aligned = aligned and img % 4 == 0
    tma_job = tma and img % 256 == 0
    full = "/tma" if tma_job else ""     # a vectorised pass over the whole input
    two = B > 1 and aligned              # mean_scratch exists wherever a routine reads it
    if mode == "autocorr":
        if aligned and W % 4 == 0:
            return ("AcVec/tma",) if tma_job else ("AcVec", "AcEdges")
        return (("Mean" + full,) if two else ()) + ("AcScalar", "AcEdges")
    if mode == "flat" and (sh, sw) == (1, 1) and H * W % 4 == 0 and aligned:
        return ("FlatSub/tma",) if tma_job and paired else ("FlatVec" + full,)
    if mode == "implicit" and (kh, kw, sh, sw, ph, pw) == (3, 3, 1, 1, 1, 1) and aligned and \
            W % 4 == 0:
        return ("3x3Vec",)
    if tma_job and mode == "implicit" and (kh, kw, sh, sw, ph, pw) == (3, 3, 2, 2, 1, 1) and \
            W % 4 == 0:
        return ("S2x3/tma",)
    two = two and not (mode == "flat" and sh * sw > 1)
    return (("Mean" + full,) if two else ()) + ("Explicit" if mode == "explicit" else "Conv",)


def _table_routine(geom, B, paired=False):
    """Routines of a layer's staging-table items.  The items of explicit im2col never cross an
    im2col row, and stage_routine stages them row by row when Wout % 4 == 0 ("Explicit/rows")."""
    C, H, W, kh, kw, sh, sw, ph, pw = geom
    Wout = (W + 2 * pw - kw) // sw + 1
    return tuple("Explicit/rows" if r == "Explicit" and Wout % 4 == 0 else r
                 for r in _routine(geom, B, _tma_enabled(B), True, paired))


# every routine sequence of the staging table and of the per-layer launches, with the batch
# classes the tests must reach it with ("1": B = 1, "+": some B > 1)
EXPECTED_ROUTES = {
    ("table", ("AcVec/tma",)): "1+",
    ("table", ("AcVec", "AcEdges")): "1+",
    ("table", ("Mean/tma", "AcScalar", "AcEdges")): "+",
    ("table", ("Mean", "AcScalar", "AcEdges")): "+",
    ("table", ("AcScalar", "AcEdges")): "1",    # C % 8 = 0: B > 1 always has the batch mean
    ("table", ("FlatVec/tma",)): "1+",
    ("table", ("FlatSub/tma",)): "1+",
    ("table", ("FlatVec",)): "1+",
    ("table", ("3x3Vec",)): "1+",
    ("table", ("S2x3/tma",)): "1+",
    ("table", ("Conv",)): "1+",                 # B > 1: strided 1x1
    ("table", ("Mean/tma", "Conv")): "+",
    ("table", ("Mean", "Conv")): "+",
    ("table", ("Explicit/rows",)): "1+",        # B > 1: C*H*W % 4 != 0
    ("table", ("Explicit",)): "1+",
    ("table", ("Mean/tma", "Explicit/rows")): "+",
    ("table", ("Mean", "Explicit/rows")): "+",
    ("table", ("Mean/tma", "Explicit")): "+",
    ("table", ("Mean", "Explicit")): "+",
    ("layer", ("AcVec", "AcEdges")): "1+",
    ("layer", ("Mean", "AcScalar", "AcEdges")): "+",
    ("layer", ("AcScalar", "AcEdges")): "1+",   # B > 1: misaligned input
    ("layer", ("FlatVec",)): "1+",
    ("layer", ("3x3Vec",)): "1+",
    ("layer", ("Conv",)): "1+",
    ("layer", ("Mean", "Conv")): "+",
    ("layer", ("Explicit",)): "1+",
    ("layer", ("Mean", "Explicit")): "+",
}


# ------------------------------------------------------------------------------- helpers
_WORST = {}      # layout kind -> (worst per-element ratio, case)


@pytest.fixture(scope="module", autouse=True)
def _report_worst(request):
    yield
    if not _WORST:
        return
    lines = ["worst |got - want| / sqrt(want_ii want_jj) per layout (bar %.0e):" % TAU]
    lines += ["  %-16s %.3e  %s" % (KERNEL[k], r, c) for k, (r, c) in sorted(_WORST.items())]
    # output capture is still active in a module fixture's teardown
    cap = request.config.pluginmanager.get_plugin("capturemanager")
    with cap.global_and_fixture_disabled():
        print("\n" + "\n".join(lines))


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


def _seed(*parts):
    return zlib.crc32(repr(parts).encode())


def _features(shape, kind, seed, dtype=torch.float32):
    """Inputs that expose misplaced terms: channel c scaled by 1 + (c % 7), border rows and
    columns 3x the interior (corners 9x).  kind "relu": post-ReLU plus a positive offset;
    "signed": zero-mean, scaled by sqrt(B) so the batch mean keeps unit size."""
    B, C, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, C, H, W, device="cuda", generator=g, dtype=torch.float64)
    x = torch.relu(x) + 0.25 if kind == "relu" else x * math.sqrt(B)
    ch = 1.0 + (torch.arange(C, device="cuda", dtype=torch.float64) % 7)
    eh = torch.ones(H, device="cuda", dtype=torch.float64)
    ew = torch.ones(W, device="cuda", dtype=torch.float64)
    eh[0] = eh[-1] = 3.0
    ew[0] = ew[-1] = 3.0
    x = x * ch[:, None, None] * eh[:, None] * ew[None, :]
    return x.to(dtype).contiguous()


def _record(kind, ratio, case):
    if kind not in _WORST or ratio > _WORST[kind][0]:
        _WORST[kind] = (ratio, case)


def _check(got, want, kind, case, tau=TAU):
    """Per-element bound, relative Frobenius error and symmetry of one d x d result."""
    got = got.double()
    assert got.shape == want.shape, (case, got.shape, want.shape)
    assert torch.isfinite(got).all(), case
    s = want.diagonal().clamp_min(0).sqrt()
    den = s[:, None] * s[None, :]
    err = (got - want).abs()
    # a tap that only ever reads padding has a zero row in the reference: it must be exact
    ratio = torch.where(den > 0, err / den.clamp_min(1e-300),
                        torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    worst = float(ratio.max())
    _record(kind, worst, case)
    if worst > tau:
        i, j = divmod(int(ratio.argmax()), ratio.shape[1])
        raise AssertionError("%s: element (%d, %d) off by %.3e of sqrt(want_ii want_jj) "
                             "(got %.9g, want %.9g)" % (case, i, j, worst, float(got[i, j]),
                                                        float(want[i, j])))
    fro = rel_fro(got, want)
    assert fro < FRO, (case, fro)
    # the autocorrelation assembly rounds mirrored blocks separately: symmetric to fp32 rounding
    asym = float((got - got.t()).norm() / got.norm().clamp_min(1e-300))
    assert asym < ASYM, (case, asym)


class _HookedConv(nn.Conv2d):
    """A Conv2d whose forward returns its input: the hooks read only the input, so the pass
    under test is the same without the convolution (and without its input restrictions)."""

    def forward(self, x):
        return x


def _conv(geom):
    C, H, W, kh, kw, sh, sw, ph, pw = geom
    return _HookedConv(C, 2, (kh, kw), stride=(sh, sw), padding=(ph, pw), bias=False).cuda()


def _oracle(x, geom):
    C, H, W, kh, kw, sh, sw, ph, pw = geom
    return O.cov_conv2d(x.double(), (kh, kw), (sh, sw), (ph, pw))


class _Net(nn.Module):
    """Named convs; a forward applies the listed ones to their inputs, in the listed order."""

    def __init__(self, convs):
        super().__init__()
        self.layers = nn.ModuleDict(convs)

    def forward(self, feeds):
        for name, x in feeds:
            self.layers[name](x)


def _hooks(pkg, net, mode, stage_sms="auto"):
    hooks = pkg.CovarianceHooks(net, add_default_ignores=False, mode=mode)
    hooks.stage_sms = stage_sms
    return hooks.register()


def _pass(pkg, net, forwards, mode, stage_sms="auto"):
    hooks = _hooks(pkg, net, mode, stage_sms)
    with torch.no_grad():
        for feeds in forwards:
            net(feeds)
    hooks.remove()
    return {k[len("layers."):-len(".weight")]: v for k, v in hooks.fea_in.items()}


def _grid_forwards(geom, B, n=3):
    """n forwards of the layer under test ("x") beside the sliding-window companion ("y"):
    post-ReLU, signed, post-ReLU inputs; fp64 oracle of each layer, summed over the forwards."""
    forwards, want = [], {"y": 0.0, "x": 0.0}
    for f in range(n):
        kind = "signed" if f % 2 else "relu"
        y = _features((B,) + COMPANION[:3], kind, _seed("y", B, f))
        x = _features((B,) + geom[:3], kind, _seed(geom, B, f))
        forwards.append([("y", y), ("x", x)])
        want["y"] = want["y"] + _oracle(y, COMPANION)
        want["x"] = want["x"] + _oracle(x, geom)
    return forwards, want


def _grid_net(geom):
    return _Net({"y": _conv(COMPANION), "x": _conv(geom)})


# ----------------------------------------------------------------------- 1. the grid
@pytest.mark.gpu
@pytest.mark.parametrize("geom,B,mode,stage_sms", _cases())
def test_covariance_geometry_grid(pkg, geom, B, mode, stage_sms):
    """Three forwards through one hook set, so the pipelined pass contracts forward i - 1 next
    to the staging of forward i; every element against the fp64 oracle."""
    torch.manual_seed(0)
    net = _grid_net(geom)
    forwards, want = _grid_forwards(geom, B)
    got = _pass(pkg, net, forwards, mode, stage_sms)
    case = "%s B=%d %s/%s" % (_gid(geom), B, mode, stage_sms)
    _check(got["x"], want["x"], _layout(*geom), case)
    _check(got["y"], want["y"], "autocorr", case + " (companion)")


# ------------------------------------------------------------ deterministic-mode subset
def _det_pass(pkg, net, forwards, mode, stage_sms):
    prev = torch.are_deterministic_algorithms_enabled()
    prev_warn = torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        hooks = _hooks(pkg, net, mode, stage_sms)
        with torch.no_grad():
            for feeds in forwards:
                net(feeds)
            out = {k: v.clone() for k, v in hooks.fea_in.items()}
        hooks.remove()
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("geom,B", [pytest.param(g, max(Bs), id="%s_b%d" % (_gid(g), max(Bs)))
                                    for g, Bs, det in GRID if det])
def test_covariance_geometry_deterministic(pkg, geom, B):
    """Under torch.use_deterministic_algorithms(True): the bound above, and bitwise equality
    between two fresh passes and between the stage_sms partitions 0, 40 and "auto"."""
    torch.manual_seed(0)
    net = _grid_net(geom)
    forwards, want = _grid_forwards(geom, B)
    ref = _det_pass(pkg, net, forwards, "deferred", 0)
    case = "%s B=%d deterministic" % (_gid(geom), B)
    _check(ref["layers.x.weight"], want["x"], _layout(*geom), case)
    _check(ref["layers.y.weight"], want["y"], "autocorr", case + " (companion)")
    for sms in (0, 40, "auto"):
        out = _det_pass(pkg, net, forwards, "deferred", sms)
        for k in ref:
            assert torch.equal(out[k], ref[k]), (case, sms, k)


# ------------------------------------------------------------------ dirty workspaces
DIRTY = [
    # (layer under test, a larger layer of the same layout run before it)
    ((16, 8, 16, 3, 3, 1, 1, 1, 1), (32, 20, 24, 3, 3, 1, 1, 1, 1)),   # autocorrelation, TMA
    ((136, 5, 6, 3, 3, 1, 1, 1, 1), (144, 9, 10, 3, 3, 1, 1, 1, 1)),   # autocorrelation, gather
    ((24, 7, 9, 1, 1, 1, 1, 0, 0), (32, 12, 13, 1, 1, 1, 1, 0, 0)),    # flat, row tail
    ((64, 8, 8, 1, 1, 1, 1, 0, 0), (64, 16, 16, 1, 1, 1, 1, 0, 0)),    # flat, TMA
    ((16, 9, 16, 3, 3, 2, 2, 1, 1), (32, 17, 32, 3, 3, 2, 2, 1, 1)),   # kStS2x3
    ((24, 7, 9, 1, 3, 1, 1, 0, 1), (32, 15, 18, 1, 3, 1, 1, 0, 1)),    # implicit
    ((16, 2, 8, 3, 3, 1, 1, 1, 1), (24, 2, 20, 3, 3, 1, 1, 1, 1)),     # implicit, kSt3x3Vec
    ((3, 7, 9, 3, 3, 1, 1, 1, 1), (5, 15, 17, 3, 3, 1, 1, 1, 1)),      # explicit
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("geom,big", [pytest.param(a, b, id=_gid(a)) for a, b in DIRTY])
def test_staging_writes_every_word_it_reads(pkg, geom, big, mode):
    """Staging must write every word the contraction reads, padding included.  A larger layer
    with inputs around 1e4 runs first; after a reset the layer under test must give its own
    result.  Immediate mode: all layers share one workspace, so the second layer stages over
    the first one's data.  Deferred / grouped: the job list changes, the first layer's workspaces
    are freed and the second layer's are allocated - this relies on the caching allocator handing
    back the freed blocks, which it does for same-stream allocations of no larger size."""
    net = _Net({"big": _conv(big), "x": _conv(geom)})
    hooks = _hooks(pkg, net, mode)
    with torch.no_grad():
        for f in range(2):                   # both job sets of the grouped modes
            net([("big", 1e4 * _features((2,) + big[:3], "relu", _seed(big, f)))])
        hooks.reset()
        want = 0.0
        for f in range(2):
            x = _features((2,) + geom[:3], "relu" if f == 0 else "signed", _seed(geom, "d", f))
            net([("x", x)])
            want = want + _oracle(x, geom)
    hooks.remove()
    fea = hooks.fea_in
    assert set(fea) == {"layers.x.weight"}
    _check(fea["layers.x.weight"], want, _layout(*geom), "%s after %s, %s" % (
        _gid(geom), _gid(big), mode))


# -------------------------------------------------- one tensor, several readers
def _readers(pkg, layers, order, B, mode):
    """Layers (name -> geometry) that all read ONE tensor, hooked in ``order``."""
    geom0 = next(iter(layers.values()))
    net = _Net({n: _conv(g) for n, g in layers.items()})
    forwards, want = [], {n: 0.0 for n in layers}
    for f in range(3):
        x = _features((B,) + geom0[:3], "signed" if f % 2 else "relu", _seed(tuple(order), B, f))
        forwards.append([(n, x) for n in order])
        for n, g in layers.items():
            want[n] = want[n] + _oracle(x, g)
    got = _pass(pkg, net, forwards, mode)
    for n, g in layers.items():
        _check(got[n], want[n], _layout(*g), "%s of %s, B=%d %s" % (n, order, B, mode))


S1 = (64, 9, 16, 1, 1, 1, 1, 0, 0)           # odd H: the subsample keeps rows 0, 2, ..., 8
S2 = (64, 9, 16, 1, 1, 2, 2, 0, 0)
AC = (16, 12, 16, 3, 3, 1, 1, 1, 1)
PAIRS = [
    ("s1_then_s2", {"s1": S1, "s2": S2}, ["s1", "s2"]),
    ("s2_then_s1", {"s1": S1, "s2": S2}, ["s2", "s1"]),
    ("two_s2", {"s1": S1, "a": S2, "b": S2}, ["a", "s1", "b"]),
    ("same_geometry", {"a": AC, "b": AC}, ["a", "b"]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("B", [1, 2])
@pytest.mark.parametrize("layers,order", [pytest.param(l, o, id=n) for n, l, o in PAIRS])
def test_one_tensor_several_readers(pkg, layers, order, B, mode):
    """A 1x1 s1 and a 1x1 s2 reader at odd H (the s2 operand is written by the s1 job's
    staging), in either hook order; two s2 readers (the second is aliased to the first, which is
    the one paired); two layers of identical geometry (staged once)."""
    _readers(pkg, layers, order, B, mode)


# ------------------------------------------------------------- deferred-mode fallbacks
MISALIGNED = [
    (16, 8, 16, 3, 3, 1, 1, 1, 1),           # autocorrelation
    (16, 9, 13, 3, 3, 1, 1, 1, 1),
    (64, 8, 8, 1, 1, 1, 1, 0, 0),            # flat
    (16, 2, 8, 3, 3, 1, 1, 1, 1),            # implicit 3x3 (kSt3x3Vec when aligned)
    (16, 9, 16, 3, 3, 2, 2, 1, 1),           # implicit 3x3 s2
    (3, 16, 16, 3, 3, 1, 1, 1, 1),           # explicit
]
MISALIGNED_BS = (1, 3)


def _misaligned(x):
    """A contiguous copy of x that starts 4 bytes into its buffer."""
    buf = torch.empty(x.numel() + 4, dtype=x.dtype, device=x.device)
    y = buf[1:1 + x.numel()].view(x.shape)
    y.copy_(x)
    assert y.is_contiguous() and y.data_ptr() % 16 != 0
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("B", MISALIGNED_BS)
@pytest.mark.parametrize("geom", [pytest.param(g, id=_gid(g)) for g in MISALIGNED])
def test_misaligned_input(pkg, geom, B, mode):
    """An input 4 bytes into its buffer: deferred mode stages it (and its forward) per layer,
    the staging routines take their unaligned forms."""
    net = _Net({"x": _conv(geom), "y": _conv(COMPANION)})
    forwards, want = [], {"x": 0.0, "y": 0.0}
    for f in range(3):
        kind = "signed" if f % 2 else "relu"
        x = _misaligned(_features((B,) + geom[:3], kind, _seed(geom, "m", B, f)))
        y = _features((B,) + COMPANION[:3], kind, _seed("y", "m", B, f))
        forwards.append([("x", x), ("y", y)])
        want["x"] = want["x"] + _oracle(x, geom)
        want["y"] = want["y"] + _oracle(y, COMPANION)
    got = _pass(pkg, net, forwards, mode)
    case = "%s misaligned B=%d %s" % (_gid(geom), B, mode)
    _check(got["x"], want["x"], _layout(*geom), case)
    _check(got["y"], want["y"], "autocorr", case + " (companion)")


RAGGED = [(16, 8, 16, 3, 3, 1, 1, 1, 1), (64, 8, 8, 1, 1, 1, 1, 0, 0),
          (16, 9, 16, 3, 3, 2, 2, 1, 1), (3, 16, 16, 3, 3, 1, 1, 1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("geom", [pytest.param(g, id=_gid(g)) for g in RAGGED])
def test_two_batch_sizes_in_one_forward(pkg, geom, mode):
    """One layer reads x (B = 3), another x[:1]: deferred mode stages the forward per layer."""
    net = _Net({"all": _conv(geom), "first": _conv(geom)})
    forwards, want = [], {"all": 0.0, "first": 0.0}
    for f in range(3):
        x = _features((3,) + geom[:3], "signed" if f % 2 else "relu", _seed(geom, "r", f))
        forwards.append([("all", x), ("first", x[:1])])
        want["all"] = want["all"] + _oracle(x, geom)
        want["first"] = want["first"] + _oracle(x[:1], geom)
    got = _pass(pkg, net, forwards, mode)
    for k in want:
        _check(got[k], want[k], _layout(*geom), "%s %s %s" % (_gid(geom), k, mode))


# ------------------------------------------------------------------------ input forms
FORMS = [
    (16, 12, 16, 3, 3, 1, 1, 1, 1),          # autocorrelation
    (16, 9, 13, 3, 3, 2, 2, 1, 1),           # implicit
    (64, 7, 9, 1, 1, 1, 1, 0, 0),            # flat
    (3, 17, 20, 7, 7, 2, 2, 3, 3),           # explicit (stem)
]


def _form(x, form):
    if form in ("float16", "bfloat16"):
        return x.to(getattr(torch, form))
    if form == "channels_last":
        y = x.to(memory_format=torch.channels_last)
        assert not y.is_contiguous()
        return y
    # "slice": every other channel of a tensor twice as wide
    B, C, H, W = x.shape
    wide = torch.zeros(B, 2 * C, H, W, device=x.device, dtype=x.dtype)
    wide[:, ::2] = x
    y = wide[:, ::2]
    assert not y.is_contiguous()
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("form", ["float16", "bfloat16", "channels_last", "slice"])
@pytest.mark.parametrize("geom", [pytest.param(g, id=_gid(g)) for g in FORMS])
def test_input_forms(pkg, geom, form, mode):
    """Half-precision inputs (against the oracle of the same values in fp64), a channels_last
    input and a non-contiguous slice."""
    net = _Net({"x": _conv(geom)})
    forwards, want = [], 0.0
    for f in range(2):
        x = _form(_features((2,) + geom[:3], "signed" if f % 2 else "relu", _seed(geom, form, f)),
                  form)
        forwards.append([("x", x)])
        want = want + _oracle(x, geom)
    got = _pass(pkg, net, forwards, mode)
    _check(got["x"], want, _layout(*geom), "%s %s %s" % (_gid(geom), form, mode))


# ----------------------------------------------------------- update_cov and Linear
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("N", [1, 5, 333])
@pytest.mark.parametrize("d", [3, 100, 130])
def test_update_cov_rows(pkg, d, N, mode):
    """update_cov(rows, key): rows (N, d) -> fea_in[key] += rows^T rows (explicit layout)."""
    net = _Net({"x": _conv((8, 4, 4, 1, 1, 1, 1, 0, 0))})
    hooks = _hooks(pkg, net, mode)
    want = 0.0
    for f in range(2):
        rows = _features((1, N, 1, d), "signed" if f else "relu", _seed("rows", d, N, f))[0, :, 0]
        hooks.update_cov(rows, "foreign.weight")
        want = want + O.gram(rows.double())
    hooks.remove()
    fea = hooks.fea_in
    assert set(fea) == {"foreign.weight"}
    _check(fea["foreign.weight"], want, "explicit", "update_cov d=%d N=%d %s" % (d, N, mode))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
@pytest.mark.parametrize("shape", [(5, 130), (4, 3), (3, 7, 130), (2, 5, 3)],
                         ids=["2d_d130", "2d_d3", "3d_d130", "3d_d3"])
def test_linear_inputs(pkg, shape, mode):
    """A Linear with d % 4 != 0; a (B, T, d) input keeps T rows of the batch mean."""
    d = shape[-1]
    lin = nn.Linear(d, 4).cuda()
    net = nn.Sequential(lin)
    hooks = pkg.CovarianceHooks(net, add_default_ignores=False, mode=mode).register()
    want = 0.0
    with torch.no_grad():
        for f in range(2):
            g = torch.Generator(device="cuda").manual_seed(_seed(shape, f))
            x = torch.randn(*shape, device="cuda", generator=g)
            x = torch.relu(x) + 0.25 if f == 0 else x
            net(x)
            want = want + O.gram(x.double().mean(dim=0).reshape(-1, d))
    hooks.remove()
    _check(hooks.fea_in["0.weight"], want, "linear", "Linear %s %s" % (shape, mode))


# ------------------------------------------------------------- one key, several extents
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
def test_one_key_several_extents_narrow_map(pkg, mode):
    """One 3x3 module at 12 x 16 and 10 x 13 (autocorrelation layout) and at 9 x 2 (W < 3: the
    generic layout, a second accumulator summed on read)."""
    geom = (16, 0, 0, 3, 3, 1, 1, 1, 1)
    net = _Net({"x": _conv(geom)})
    forwards, want = [], 0.0
    for f in range(2):
        feeds = []
        for H, W in ((12, 16), (9, 2), (10, 13)):
            x = _features((2, 16, H, W), "signed" if f else "relu", _seed("ext", H, W, f))
            feeds.append(("x", x))
            want = want + _oracle(x, geom)
        forwards.append(feeds)
    got = _pass(pkg, net, forwards, mode)
    _check(got["x"], want, "autocorr", "several extents %s" % mode)


# ------------------------------------------------------------- 5. routes (no GPU)
def _route_cases():
    """(route, geometry, B, aligned, paired) of every staged layer the GPU tests above run: route
    "table" (deferred mode's staging table) or "layer" (the per-layer launches)."""
    out = []
    for geom, Bs, _det in GRID:
        for B in Bs:
            out += [("table", geom, B, True, False), ("layer", geom, B, True, False),
                    ("table", COMPANION, B, True, False), ("layer", COMPANION, B, True, False)]
    for geom in MISALIGNED:
        for B in MISALIGNED_BS:
            out.append(("layer", geom, B, False, False))     # also deferred mode's fallback
    for geom in RAGGED:
        out += [("layer", geom, 3, True, False), ("layer", geom, 1, True, False)]
    for _name, layers, order in PAIRS:
        for B in (1, 2):
            full = [g for g in layers.values() if g[5:7] == (1, 1)]
            for g in layers.values():
                paired = bool(full) and g is full[0] and any(
                    _sub_pair_ok(s, g, B) for s in layers.values() if s[5:7] == (2, 2))
                sibling = g[5:7] == (2, 2) and full and _sub_pair_ok(g, full[0], B)
                if not sibling:
                    out.append(("table", g, B, True, paired))
                out.append(("layer", g, B, True, False))
    return out


def test_every_staging_route_is_reached():
    """The layer geometries, batch sizes and input alignments of this file reach every routine
    sequence that plan_stage_job can pick for a staging table and for the per-layer launches,
    each with B = 1 and with some B > 1 where the planner allows it (EXPECTED_ROUTES)."""
    reached = {}
    for route, geom, B, aligned, paired in _route_cases():
        seq = _table_routine(geom, B, paired) if route == "table" else \
            _routine(geom, B, tma=False, aligned=aligned)
        reached.setdefault((route, seq), set()).add("1" if B == 1 else "+")
    unknown = set(reached) - set(EXPECTED_ROUTES)
    assert not unknown, unknown
    missing = {k: v for k, v in EXPECTED_ROUTES.items() if not set(v) <= reached.get(k, set())}
    assert not missing, missing


def test_restated_layout_matches_the_library():
    """_layout above agrees with the layout nsgp_cov_conv2d_layout reports for every geometry of
    this file (autocorrelation kind; taps and internal rows of the other three)."""
    import ctypes
    from nsgp_repre_b200._lib import lib, CovLayout
    geoms = {g for g, _Bs, _det in GRID} | set(MISALIGNED) | set(RAGGED) | set(FORMS) | \
        {g for _n, layers, _o in PAIRS for g in layers.values()} | \
        {g for pair in DIRTY for g in pair} | {COMPANION}
    for geom in sorted(geoms):
        L = CovLayout()
        assert lib.nsgp_cov_conv2d_layout(*geom, ctypes.byref(L)) == 0, geom
        C, H, W, kh, kw = geom[:5]
        mode = _layout(*geom)
        assert (L.kind == 1) == (mode == "autocorr"), geom
        assert L.d == C * kh * kw, geom
        if mode == "flat":
            assert (L.taps, L.d_int) == (1, C), geom
        elif mode == "implicit":
            assert (L.taps, L.d_int) == (kh * kw, kh * kw * C), geom
        elif mode == "explicit":
            assert (L.taps, L.d_int) == (1, -(-C * kh * kw // 8) * 8), geom
