"""``torch.use_deterministic_algorithms(True)``: the training path (covariance pass, projected
step, prototype build, EWC penalty) gives bitwise identical results for identical inputs, and
the entry points without a deterministic form raise (warn under ``warn_only=True``).

The switch is turned on only around library calls (``_det``), so the fp64 oracle's own
matmuls run as usual.  Under the switch torch's own cuBLAS calls need a workspace config; the
Linear forwards of the covariance model are such calls.
"""
import contextlib
import os
import warnings

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import rel_fro
from oracle import restated as O
from oracle import synth

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

TOL = 1e-4


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


@contextlib.contextmanager
def _det(on=True, warn_only=False):
    prev = torch.are_deterministic_algorithms_enabled()
    prev_warn = torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


# ------------------------------------------------------------------------------ CPU
def test_deterministic_symbols_and_size_queries():
    """The switch is exported and the size queries grow only while it is set; they stay
    host-only (no device is needed to call them)."""
    import ctypes
    from nsgp_repre_b200._lib import lib, CovLayout, CovJob
    assert lib.nsgp_get_deterministic() in (0, 1)
    prev = lib.nsgp_set_deterministic(0)
    try:
        def sizes():
            out = {}
            for name, geom in (("1x1", (64, 200, 336, 1, 1, 1, 1, 0, 0)),
                               ("3x3s1", (64, 100, 168, 3, 3, 1, 1, 1, 1)),
                               ("3x3s2", (64, 100, 168, 3, 3, 2, 2, 1, 1))):
                L = CovLayout()
                assert lib.nsgp_cov_conv2d_layout(*geom, ctypes.byref(L)) == 0
                out[name] = (L.workspace_bytes, L.acc_bytes)
                jobs = (CovJob * 2)()
                for j in jobs:
                    (j.Cin, j.H, j.W, j.kh, j.kw, j.sh, j.sw, j.ph, j.pw) = geom
                    j.acc, j.workspace, j.workspace_bytes = 1 << 20, 1 << 30, L.workspace_bytes
                out[name + "/group"] = lib.nsgp_cov_group_bytes(jobs, 2)
            out["repre"] = lib.repre_build_prototypes_workspace_bytes(400, 12544, 4, 9)
            out["repre_small"] = lib.repre_build_prototypes_workspace_bytes(400, 1024, 4, 9)
            out["ewc"] = lib.nsgp_ewc_table_bytes(5)
            return out
        off = sizes()
        assert lib.nsgp_set_deterministic(1) == 0
        assert lib.nsgp_get_deterministic() == 1
        on = sizes()
        assert lib.nsgp_set_deterministic(0) == 1
        assert sizes() == off
    finally:
        lib.nsgp_set_deterministic(prev)
    for k in off:
        if k.endswith("/group") or k in ("ewc", "repre"):
            assert on[k] > off[k], k
    for k in ("1x1", "3x3s1", "3x3s2"):
        assert on[k][0] > off[k][0] and on[k][1] == off[k][1], k
    # a Gram of one K chain per tile needs no slots
    assert on["repre_small"] == off["repre_small"]


# ------------------------------------------------------------------------ covariance
class _CovNet(nn.Module):
    """Long-K layers: a 1x1 conv at 200x336, the 7x7 stride-2 stem, a 3x3 stride-1
    (sliding-window) and a 3x3 stride-2 conv, one 3x3 conv hooked at five extents (one of them
    under 3 px, i.e. a second accumulator layout) and a Linear."""

    def __init__(self):
        super().__init__()
        self.lateral = nn.Conv2d(16, 32, 1)
        self.stem = nn.Conv2d(16, 32, 7, 2, 3)
        self.s1 = nn.Conv2d(32, 32, 3, 1, 1)
        self.s2 = nn.Conv2d(32, 64, 3, 2, 1)
        self.shared = nn.Conv2d(64, 32, 3, 1, 1)
        self.fc = nn.Linear(64, 16)

    def forward(self, x):
        self.lateral(x)
        y = self.s2(self.s1(self.stem(x)))
        for size in ((50, 84), (25, 42), (13, 21), (7, 11), (2, 2)):
            self.shared(F.adaptive_avg_pool2d(y, size))
        self.fc(y.mean(dim=(2, 3)))
        return y


def _cov_inputs():
    g = torch.Generator().manual_seed(5)
    return [torch.randn(2, 16, 200, 336, generator=g) for _ in range(3)]


def _cov_pass(pkg, net, xs, mode, stage_sms="auto"):
    hooks = pkg.CovarianceHooks(net, mode=mode, add_default_ignores=False)
    hooks.stage_sms = stage_sms
    hooks.register()
    with _det(), torch.no_grad():
        for x in xs:
            net(x)
        out = {k: v.clone() for k, v in hooks.fea_in.items()}
    hooks.remove()
    return out


def _oracle_of_device_inputs(net, xs):
    """fp64 covariances of the layer inputs the device forward produces.  The inputs of the
    layers behind the first conv depend on cuDNN's arithmetic (TF32 convolutions by default),
    so a CPU forward would feed the oracle different inputs; the hooks capture the device's."""
    names = {m: n for n, m in net.named_modules()}
    fea = {}

    def hook(m, inputs, _out):
        x = inputs[0].detach().double().cpu()
        key = names[m] + ".weight"
        if isinstance(m, nn.Linear):
            O.accumulate(fea, key, O.cov_linear(x))
        else:
            O.accumulate(fea, key, O.cov_conv2d(x, m.kernel_size, m.stride, m.padding))

    handles = [m.register_forward_hook(hook) for m in net.modules()
               if isinstance(m, (nn.Conv2d, nn.Linear))]
    with _det(), torch.no_grad():
        for x in xs:
            net(x)
    for h in handles:
        h.remove()
    return fea


@pytest.fixture(scope="module")
def cov_case():
    torch.manual_seed(0)
    net = _CovNet().eval().cuda()
    xs = [x.cuda() for x in _cov_inputs()]
    return net, xs, _oracle_of_device_inputs(net, xs)


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), k


def _close(got, want):
    assert got.keys() == want.keys()
    for k in got:
        err = rel_fro(got[k], want[k])
        assert err < TOL, (k, err)


@pytest.mark.gpu
def test_deferred_pass_is_bitwise_reproducible(pkg, cov_case):
    """Three forwards per pass; every stage_sms partition and two fresh hook sets agree."""
    net, xs, want = cov_case
    ref = _cov_pass(pkg, net, xs, "deferred", 0)
    _close(ref, want)
    for sms in (0, 40, "auto"):
        _same(_cov_pass(pkg, net, xs, "deferred", sms), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["grouped", "immediate"])
def test_grouped_and_immediate_passes_are_bitwise_reproducible(pkg, cov_case, mode):
    net, xs, want = cov_case
    a = _cov_pass(pkg, net, xs, mode)
    _close(a, want)
    _same(_cov_pass(pkg, net, xs, mode), a)


@pytest.mark.gpu
def test_switching_on_after_two_forwards_rebuilds_the_tables(pkg, cov_case):
    """Two forwards with the switch off, a reset, then three with it on, through one hook set:
    the tables of the other mode are rebuilt, and the result is the one of a fresh pass."""
    net, xs, want = cov_case
    ref = _cov_pass(pkg, net, xs, "deferred")
    for _ in range(2):
        hooks = pkg.CovarianceHooks(net, mode="deferred", add_default_ignores=False)
        hooks.register()
        with torch.no_grad():
            for x in xs[:2]:
                net(x)
            hooks.reset()
            with _det():
                for x in xs:
                    net(x)
                out = {k: v.clone() for k, v in hooks.fea_in.items()}
        hooks.remove()
        _same(out, ref)


# --------------------------------------------------------------------------- step
def _householder_eigens(d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    v = torch.randn(d, 1, dtype=torch.float64, device="cuda", generator=g)
    h = torch.eye(d, dtype=torch.float64, device="cuda")
    h.addmm_(v, v.t(), alpha=-2.0 / float(v.square().sum()))
    i = torch.arange(d, dtype=torch.float64)
    m = d // 2
    spec = torch.where(i < m, 2.0 - i / m, 1e-2 * torch.exp(-4.0 * (i - m) / (d - m)))
    return {"eigen_value": spec.float().cuda(), "eigen_vector": h.float()}


STEP_LAYERS = [
    ("backbone.layer3.0.conv2.weight", (256, 128, 3, 3)),
    ("neck.fpn_convs.0.conv.weight", (256, 256, 3, 3)),
    ("rpn_head.rpn_cls.weight", (3, 256, 1, 1)),
    ("roi_head.bbox_head.fc_cls.weight", (21, 1024)),
    ("backbone.conv1.weight", (64, 3, 7, 7)),
    ("roi_head.bbox_head.shared_fcs.0.weight", (64, 12544)),
]


def _step_run(pkg, ratio, params0, grads, transforms=None):
    names = [n for n, _ in STEP_LAYERS]
    params = [nn.Parameter(p.clone()) for p in params0]
    opt = pkg.SGDNSCL(params, svd=True, lr=0.02, momentum=0.9, weight_decay=1e-4, nesterov=True)
    opt.lowrank_max_ratio = ratio
    opt.param_groups[0]["names"] = names
    for k, (n, shape) in enumerate(STEP_LAYERS):
        opt.eigens[n] = _householder_eigens(params[k].numel() // shape[0], 11 + k)
    opt.get_transforms()
    with _det():
        for it in range(3):
            for p, g in zip(params, grads[it]):
                p.grad = g.clone()
            opt.step()
    bufs = [opt.state[p]["previous_grad"].clone() for p in params]
    return [p.detach().clone() for p in params], bufs, opt


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [1.0, 0.0], ids=["lowrank", "dense"])
def test_projected_step_is_bitwise_reproducible(pkg, ratio):
    """Three Nesterov steps of a protected set (with a d = 12 544 layer) twice from cloned
    state: weights and momentum bitwise equal, and within the step bar of the fp64 oracle."""
    g = torch.Generator(device="cuda").manual_seed(3)
    params0 = [0.01 * torch.randn(s, device="cuda", generator=g) for _, s in STEP_LAYERS]
    grads = [[torch.randn(s, device="cuda", generator=g) for _, s in STEP_LAYERS]
             for _ in range(3)]
    w1, b1, opt = _step_run(pkg, ratio, params0, grads)
    assert (opt._plans[0]["t_arena"] is not None) == (ratio > 0)      # the form that ran
    w2, b2, _ = _step_run(pkg, ratio, params0, grads)
    for a, b in zip(w1 + b1, w2 + b2):
        assert torch.equal(a, b)
    names = [n for n, _ in STEP_LAYERS]
    ref = {n: p.double() for n, p in zip(names, params0)}
    states = {}
    for it in range(3):
        O.sgd_nscl_step(ref, {n: gr.double() for n, gr in zip(names, grads[it])}, states,
                        {n: opt.transforms[n].double() for n in names}, svd=True, lr=0.02,
                        momentum=0.9, weight_decay=1e-4, nesterov=True)
    for n, w in zip(names, w1):
        assert rel_fro(w - params0[names.index(n)], ref[n] - params0[names.index(n)].double()) \
            < TOL, n


# ------------------------------------------------------------------------ prototypes
def _masks_equal(a, b):
    assert len(a) == len(b)
    for ma, mb in zip(a, b):
        assert len(ma) == len(mb)
        for x, y in zip(ma, mb):
            assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("classes,per_class", [(10, 60), (40, 30)], ids=["voc10", "coco40"])
def test_prototype_build_is_bitwise_reproducible(pkg, classes, per_class):
    """Two builds (and a graph-replayed third and fourth), without and with replayed masks."""
    feats, lab = synth.proto_features(seed=21, classes=classes, per_class=per_class, D=12544,
                                      bg=40)
    f_d, l_d = feats.cuda(), lab.cuda()
    want_p, want_l, _ = O.build_prototypes(feats, lab, range(classes), 10)
    runs = []
    with _det():
        for _ in range(2):
            mp = pkg.MultiPrototypeReplay(10).build(f_d, l_d, range(classes))
            runs.append((mp.bbox_featss.clone(), mp.tmp_label.clone(), mp.save_idx))
        mp = pkg.MultiPrototypeReplay(10)
        for run in range(4):
            mp.build(f_d, l_d, range(classes))
            assert (mp._graph is not None) == (run >= 1)
            runs.append((mp.bbox_featss.clone(), mp.tmp_label.clone(), mp.save_idx))
    for p, l, m in runs[1:]:
        assert torch.equal(p, runs[0][0]) and torch.equal(l, runs[0][1])
        _masks_equal(m, runs[0][2])
    assert torch.equal(runs[0][1].cpu(), want_l)
    assert rel_fro(runs[0][0], want_p) < 1e-5
    # replayed mask.pth
    saved = runs[0][2]
    again = []
    with _det():
        for _ in range(2):
            mp = pkg.MultiPrototypeReplay(10).build(f_d, l_d, range(classes), saved_masks=saved)
            again.append((mp.bbox_featss.clone(), mp.tmp_label.clone(), mp.save_idx))
    assert torch.equal(again[0][0], again[1][0]) and torch.equal(again[0][1], again[1][1])
    _masks_equal(again[0][2], again[1][2])


# ------------------------------------------------------------------------------- EWC
class _Tiny(nn.Module):
    def __init__(self):
        super().__init__()
        self.bn = nn.BatchNorm2d(3000)
        self.conv = nn.Conv2d(64, 64, 3)

    def loss(self, *a, **k):
        return {}


@pytest.mark.gpu
def test_ewc_penalty_is_bitwise_reproducible(pkg):
    torch.manual_seed(2)
    net = _Tiny().cuda()
    reg = {n: p for n, p in net.named_parameters()}
    terms = {"importance": {n: [torch.rand(2, *p.shape, device="cuda")] for n, p in reg.items()},
             "task_param": {n: [p.detach() + 0.1 * torch.randn(2, *p.shape, device="cuda")]
                            for n, p in reg.items()}}
    hook = pkg.EWCHook(module=net, reg_params=reg, ewc_reg_terms=terms)
    out = []
    with _det():
        for _ in range(2):
            for p in reg.values():
                p.grad = None
            loss = hook.penalty()
            loss.backward()
            out.append((loss.detach().clone(), [p.grad.clone() for p in reg.values()]))
    assert torch.equal(out[0][0], out[1][0])
    for a, b in zip(out[0][1], out[1][1]):
        assert torch.equal(a, b)
    want = O.ewc_penalty({n: p.detach().cpu().requires_grad_() for n, p in reg.items()},
                         {k: {n: [t.cpu() for t in v] for n, v in d.items()}
                          for k, d in terms.items()})
    assert abs(float(out[0][0]) - float(want)) <= 1e-5 * abs(float(want))


# --------------------------------------------------------------------------- raising
def _roi_case(pkg):
    feats, rois, labels = synth.roi_case(4, batch=2, channels=16, img_h=128, img_w=160,
                                         n_rois=64, classes=5, strides=(4, 8))
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=0),
                                 out_channels=16, featmap_strides=[4, 8])
    return ext, [f.cuda() for f in feats], rois.cuda(), labels.cuda()


@pytest.mark.gpu
def test_entries_without_a_deterministic_form_raise(pkg):
    ext, feats, rois, labels = _roi_case(pkg)
    fg = [f.clone().requires_grad_() for f in feats]
    x = torch.randn(50, 64, device="cuda")
    c0 = x[:4].clone()

    def calls():
        yield "class_sums", lambda: ext.class_sums(feats, rois, labels, 5)
        yield "roi_align_backward", lambda: ext(fg, rois).sum().backward()
        yield "kmeans", lambda: pkg.kmeans_prototypes(x, c0, iters=2)

    for name, fn in calls():
        fn()                                          # switch off: runs as before
        with _det():
            with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
                fn()
        with _det(warn_only=True):
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                fn()
            assert any("deterministic implementation" in str(m.message) for m in w), name
    # RoIAlign forward without class sums is per element: allowed
    with _det():
        a = ext(feats, rois)
        b = ext(feats, rois)
    assert torch.equal(a, b)
