"""GPU parity tests: the CUDA path (through the C ABI) against the oracle
restatement and the golden fixtures produced by the reference's own functions.

Tolerances (BASELINE.json north_star): covariances, projectors, projected updates
and prototypes within 1e-4 relative Frobenius error; neighbour masks identical
except for documented near-ties (|S - 0.6| < 1e-5); integer / index results
bit-exact.
"""
import os

import pytest
import torch

from conftest import rel_fro
from oracle import restated as O
from oracle import synth

pytestmark = pytest.mark.gpu

TOL = 1e-4
# 3xTF32 on tcgen05: operands carry ~21 mantissa bits and the tensor core accumulates
# with truncation (~2^-25.6 relative per accumulate step, measured on B200); the K
# chain per TMEM accumulator is bounded to 32 K-blocks (384 steps) -> <= ~1e-5.
ENGINE_TOL = 2e-5


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), map_location="cpu", weights_only=False)


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


@pytest.fixture(params=[0, 1], ids=["tcgen05", "simt"])
def engine(request, pkg):
    """The shipped library has ONE engine (tcgen05); the SIMT cross-check engine exists only in
    the bring-up build (make BRINGUP=1, NSGP_BRINGUP_LIB=1)."""
    if not pkg._lib.HAS_BRINGUP:
        if request.param != 0:
            pytest.skip("SIMT cross-check engine: bring-up build only")
        yield 0
        return
    prev = pkg._lib.lib.nsgp_set_engine(request.param)
    yield request.param
    pkg._lib.lib.nsgp_set_engine(prev)


def _stream():
    return torch.cuda.current_stream().cuda_stream


# --------------------------------------------------------------------------- engine
@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (128, 128, 256), (200, 136, 100),
                                   (64, 8, 36), (384, 640, 1056), (8, 8, 4), (130, 300, 3076)])
def test_contraction_gemm_3xtf32(pkg, engine, M, N, K):
    """C += A B^T on the selected engine vs fp64; 3xTF32 must be fp32-faithful."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    B = torch.randn(N, K, device="cuda", generator=g)
    C0 = torch.randn(M, N + (-N) % 4, device="cuda", generator=g)
    ah, al, bh, bl = (torch.empty_like(A), torch.empty_like(A), torch.empty_like(B),
                      torch.empty_like(B))
    pkg._lib.check(lib.nsgp_split_tf32(ptr(A), ptr(ah), ptr(al), A.numel(), _stream()), "split")
    pkg._lib.check(lib.nsgp_split_tf32(ptr(B), ptr(bh), ptr(bl), B.numel(), _stream()), "split")
    assert torch.equal((ah.view(torch.int32) & 0x1FFF), torch.zeros_like(ah, dtype=torch.int32))
    C = C0.clone()
    pkg._lib.check(lib.nsgp_gemm_nt(ptr(ah), ptr(al), ptr(bh), ptr(bl), M, N, K, ptr(C),
                                          C.shape[1], _stream()), "gemm")
    want = C0.double()
    want[:, :N] += A.double() @ B.double().t()
    assert rel_fro(C[:, :N], want[:, :N]) < ENGINE_TOL
    assert torch.equal(C[:, N:], C0[:, N:])          # padding columns untouched


# ----------------------------------------------------------------------- covariance
@pytest.mark.parametrize("mode", ["deferred", "grouped", "immediate"])
def test_covariance_toy_model_matches_reference_fixture(pkg, engine, golden_dir, mode):
    """Every conv geometry of R50-FPN at toy size, 3 batches, through the forward
    hooks, against the fixture produced by the reference's compute_cov/update_cov."""
    g = _load(golden_dir, "cov_toy.pt")
    net = synth.ToyDetector()
    net.load_state_dict(g["state_dict"])
    batches = synth.toy_batches(seed=g["seed"])
    net = net.cuda()
    if engine != 0 and mode != "deferred":
        pytest.skip("the bring-up engine has one host mode")
    hooks = pkg.CovarianceHooks(net, add_default_ignores=False, mode=mode)
    fea = hooks.cal_fea_in([b.cuda() for b in batches])
    assert set(fea) == set(g["fea_in"])
    for k, ref in g["fea_in"].items():
        assert fea[k].shape == ref.shape
        assert rel_fro(fea[k], ref) < TOL, k
        assert rel_fro(fea[k], fea[k].t()) == 0.0          # exactly symmetric


GEOMS = [
    # (Cin, H, W, k, s, p, B)                      what it stands for
    (64, 40, 56, 3, 1, 1, 2),     # layer1 conv2: 9 taps x 64 rows, tiles span taps
    (128, 31, 45, 3, 2, 1, 3),    # layerN.0 conv2: stride-2 phases, odd extent
    (256, 25, 42, 3, 1, 1, 1),    # fpn conv at P5-like extent (Wout not /32)
    (256, 50, 84, 1, 1, 0, 2),    # 1x1 flat
    (512, 25, 42, 1, 2, 0, 2),    # downsample 1x1 s2
    (3, 64, 96, 7, 2, 3, 2),      # stem, explicit im2col, d = 147
    (64, 17, 23, 1, 1, 0, 4),     # d = 64 < one tile
    (8, 9, 11, 3, 1, 1, 2),       # tiny
    (16, 3, 3, 3, 1, 1, 2),       # smallest map the autocorrelation layout takes
    (24, 12, 16, 3, 1, 1, 3),     # W % 4 == 0: vectorised autocorrelation staging, Cin = 24
    (8, 2, 9, 3, 1, 1, 2),        # H < 3: falls back to the tap-pair layout
    (16, 12, 40, 5, 1, 2, 2),     # 25 taps -> explicit fallback
]


@pytest.mark.parametrize("mode", ["deferred", "grouped"])
@pytest.mark.parametrize("Cin,H,W,k,s,p,B", GEOMS)
def test_covariance_layer_geometries(pkg, engine, Cin, H, W, k, s, p, B, mode):
    if engine != 0 and mode != "deferred":
        pytest.skip("the bring-up engine has one host mode")
    g = torch.Generator().manual_seed(Cin * 131 + H)
    conv = torch.nn.Conv2d(Cin, 4, k, stride=s, padding=p, bias=False).cuda()
    model = torch.nn.Sequential(conv)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False, mode=mode).register()
    want = None
    for _ in range(2):
        x = torch.relu(torch.randn(B, Cin, H, W, generator=g))
        with torch.no_grad():
            model(x.cuda())
        c = O.cov_conv2d(x.double(), (k, k), (s, s), (p, p))
        want = c if want is None else want + c
    hooks.remove()
    got = hooks.fea_in["0.weight"]
    assert got.shape == (Cin * k * k, Cin * k * k)
    assert rel_fro(got, want) < 2e-5


def test_covariance_deferred_rejects_inplace_modification(pkg, engine):
    """Deferred staging reads the layer input at the end of the forward: an in-place
    write between the hook and the flush must be an error, never a wrong covariance."""
    if engine != 0:
        pytest.skip("grouped launches need the tcgen05 engine")

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = torch.nn.Conv2d(8, 4, 1, bias=False)

        def forward(self, x):
            y = self.conv(x)
            x.mul_(2.0)
            return y

    net = Net().cuda()
    x = torch.relu(torch.randn(2, 8, 6, 8)).cuda()
    hooks = pkg.CovarianceHooks(net, add_default_ignores=False, mode="deferred").register()
    with pytest.raises(pkg._lib.NsgpError, match="modified in place"):
        with torch.no_grad():
            net(x.clone())
    hooks.remove()
    hooks2 = pkg.CovarianceHooks(net, add_default_ignores=False, mode="grouped").register()
    with torch.no_grad():
        net(x.clone())
    hooks2.remove()
    want = O.cov_conv2d(x.cpu().double(), (1, 1), (1, 1), (0, 0))
    assert rel_fro(hooks2.fea_in["conv.weight"], want) < 2e-5


FULL_SIZE = [
    # (Cin, H, W, k, s, p)  BASELINE configs[1] extents (800x1344 input)
    (64, 200, 336, 3, 1, 1),      # layer1 conv2: autocorrelation layout, 67 200 positions
    (256, 200, 336, 3, 1, 1),     # fpn_convs.0: d = 2304, the heaviest layer
    (128, 200, 336, 3, 2, 1),     # layer2.0 conv2: stride-2 tap-pair layout
    (256, 200, 336, 1, 1, 0),     # 1x1 flat
    (3, 800, 1344, 7, 2, 3),      # stem, explicit im2col
    (512, 25, 42, 3, 1, 1),       # layer4 conv2: W % 4 != 0 (scalar autocorrelation staging)
]


@pytest.mark.parametrize("Cin,H,W,k,s,p", FULL_SIZE)
def test_covariance_full_size_properties(pkg, Cin, H, W, k, s, p):
    """Full BASELINE extents, where the CPU oracle would take minutes: size-independent
    properties of X^T X checked against independent fp64 reductions on the device.
      * row sums:  cov @ 1 = X^T (X 1), both factors computed as convolutions of the batch mean
        (a checksum of every row of the d x d result)
      * diagonal = squared column norms of X, symmetry
      * homogeneity: inputs scaled by 2 give 4x the covariance (powers of two are exact in
        every product), accumulating two passes gives their sum"""
    import torch.nn.functional as F
    g = torch.Generator(device="cuda").manual_seed(Cin + H)
    B = 2
    x = torch.relu(torch.randn(B, Cin, H, W, device="cuda", generator=g))
    conv = torch.nn.Conv2d(Cin, 4, k, stride=s, padding=p, bias=False).cuda()
    model = torch.nn.Sequential(conv)

    def run(inputs):
        hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
        with torch.no_grad():
            for t in inputs:
                model(t)
        hooks.remove()
        return hooks.fea_in["0.weight"]

    cov = run([x])
    d = Cin * k * k
    assert cov.shape == (d, d)
    # symmetric up to fp32 rounding (mirrored blocks of the autocorrelation assembly come from
    # separately rounded edge corrections; the reference's torch.mm is not bitwise symmetric either)
    asym = float((cov - cov.t()).double().norm() / cov.double().norm())
    assert asym < 1e-6, asym
    m = x.double().mean(0, keepdim=True)                               # (1,Cin,H,W)
    ones = torch.ones(1, Cin, k, k, dtype=torch.float64, device="cuda")
    rowsum = F.conv2d(m, ones, stride=s, padding=p)[0, 0]              # X 1  per output position
    Ho, Wo = rowsum.shape
    # X^T (X 1): for (c, i, j): sum_pos m~[c][s*oy+i-p][s*ox+j-p] * rowsum[oy][ox]
    mp = F.pad(m[0], (p, p, p, p))                                     # (Cin, H+2p, W+2p)
    want = torch.empty(Cin, k, k, dtype=torch.float64, device="cuda")
    sq = torch.empty(Cin, k, k, dtype=torch.float64, device="cuda")
    for i in range(k):
        for j in range(k):
            win = mp[:, i:i + s * (Ho - 1) + 1:s, j:j + s * (Wo - 1) + 1:s]
            want[:, i, j] = (win * rowsum).sum((1, 2))
            sq[:, i, j] = (win * win).sum((1, 2))
    got = cov.double().sum(1)
    # the bar is 1e-4 (BASELINE north_star).  What is left is the tensor core's truncating fp32
    # accumulate: ~1.9e-8 relative per step, one-sided for the non-negative post-ReLU inputs,
    # times the chain length (<= 576 steps in the sliding-window kernel) ~ 1.1e-5 (DESIGN.md 4)
    assert rel_fro(got, want.reshape(-1)) < 3e-5
    assert rel_fro(torch.diagonal(cov).double(), sq.reshape(-1)) < 3e-5
    # (partial tiles of different K ranges meet in fp32 red.add, whose order varies from
    # run to run: equal up to that, not bit for bit)
    assert rel_fro(run([2.0 * x]), 4.0 * cov.double()) < 1e-6
    assert rel_fro(run([x, x]), 2.0 * cov.double()) < 1e-6


def test_prototypes_full_size_matches_oracle(pkg):
    """BASELINE configs[1] RePRE shape: M = 4096 RoIs x 12544, 19 old classes, 75 %
    background (bench.py's generator) against the CPU restatement."""
    import bench
    feats, lab = bench.synthetic_rois(8, 7)
    want_p, want_l, want_m = O.build_prototypes(feats, lab, range(19), 10)
    mp = pkg.MultiPrototypeReplay(10).build(feats.cuda(), lab.cuda(), range(19))
    assert torch.equal(mp.tmp_label.cpu(), want_l)
    for mine, ref in zip(mp.save_idx, want_m):
        assert len(mine) == len(ref)
        for a, b in zip(mine, ref):
            assert torch.equal(a.cpu().bool(), b.bool())
    assert rel_fro(mp.bbox_featss, want_p) < 1e-5
    assert torch.equal(mp.staged().cpu(), mp.bbox_featss.cpu())


def test_covariance_long_k_chain(pkg, engine):
    """N = 67 200 positions (the P2-level extent at 800x1344): exercises K splits
    and the fp32 accumulation chain."""
    g = torch.Generator().manual_seed(3)
    x = torch.relu(torch.randn(1, 64, 200, 336, generator=g)) + 0.5
    conv = torch.nn.Conv2d(64, 4, 3, padding=1, bias=False).cuda()
    model = torch.nn.Sequential(conv)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
    with torch.no_grad():
        model(x.cuda())
    hooks.remove()
    want = O.cov_conv2d(x.double(), (3, 3), (1, 1), (1, 1))
    assert rel_fro(hooks.fea_in["0.weight"], want) < 2e-5


def test_covariance_linear_and_update_cov(pkg, engine):
    g = torch.Generator().manual_seed(11)
    lin = torch.nn.Linear(200, 6).cuda()
    model = torch.nn.Sequential(lin)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
    xs = [torch.randn(5, 200, generator=g) for _ in range(3)]
    with torch.no_grad():
        for x in xs:
            model(x.cuda())
    hooks.remove()
    want = sum(O.cov_linear(x.double()) for x in xs)
    assert rel_fro(hooks.fea_in["0.weight"], want) < ENGINE_TOL
    # update_cov(rows, key): the reference's (N, d) entry point
    rows = torch.randn(333, 72, generator=g)
    hooks.update_cov(rows.cuda(), "extra.weight")
    hooks.update_cov(rows.cuda(), "extra.weight")
    assert rel_fro(hooks.fea_in["extra.weight"], 2 * O.gram(rows.double())) < ENGINE_TOL


def test_covariance_merge_previous_and_save(pkg, tmp_path):
    conv = torch.nn.Conv2d(8, 4, 3, padding=1).cuda()
    model = torch.nn.Sequential(conv)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False)
    x = torch.randn(2, 8, 10, 12)
    old = {"0.weight": torch.eye(72)}
    out = hooks.cal_fea_in([x.cuda()], previous=old, save_path=str(tmp_path / "covariance.pth"))
    want = O.cov_conv2d(x, (3, 3), (1, 1), (1, 1)) + old["0.weight"]
    assert rel_fro(out["0.weight"], want) < TOL
    again = torch.load(str(tmp_path / "covariance.pth"), map_location="cpu")
    assert set(again) == {"0.weight"} and rel_fro(again["0.weight"], want) < TOL


# ------------------------------------------------------------------------ projector
@pytest.mark.parametrize("offset", [0.0, 0.5, -0.5, 3.0])
def test_projector_matches_reference_fixture(pkg, golden_dir, offset):
    """get_eigens (GPU syevd) + get_transforms vs the reference's fp32 SVD build.
    P = V0 V0^T is compared, never the basis (sign / rotation ambiguity)."""
    g = _load(golden_dir, "projector.pt")
    ents = g["proj"][offset]
    covs = {n: synth.decaying_cov(*g["seeds"][n][:2], rank=g["seeds"][n][2]).cuda()
            for n in ents}
    params = [torch.nn.Parameter(torch.zeros(4, covs[n].shape[0], device="cuda")) for n in ents]
    opt = pkg.SGDNSCL(params, lr=0.02, svd=True)
    opt.param_groups[0]["names"] = list(ents)
    opt.get_eigens(covs)
    opt.get_transforms(offset=offset)
    for n, ent in ents.items():
        assert rel_fro(opt.eigens[n]["eigen_value"], ent["svals"]) < 1e-5
        mask = opt.adaptive_threshold(opt.eigens[n]["eigen_value"], offset=offset)
        assert int(mask.long().argmax()) == ent["i_thres"], n
        assert rel_fro(opt.transforms[n], ent["transform"]) < TOL, n


# ------------------------------------------------------------------------- SGD step
@pytest.mark.parametrize("tag", ["mom_wd", "plain", "nesterov_damp"])
def test_sgd_nscl_steps_match_reference_fixture(pkg, engine, golden_dir, tag):
    g = _load(golden_dir, "sgd_steps.pt")
    proj = _load(golden_dir, "projector.pt")["proj"][0.0]
    run = g["steps"][tag]
    names = list(g["init"])
    params = [torch.nn.Parameter(g["init"][n].clone().cuda()) for n in names]
    opt = pkg.SGDNSCL(params, svd=True, **run["kw"])
    opt.param_groups[0]["names"] = names
    for n, e in proj.items():
        opt.transforms[n] = e["transform"].cuda()
    for step, want in zip(g["grads"], run["traj"]):
        for n, p in zip(names, params):
            p.grad = step[n].clone().cuda()
        opt.step()
        for n, p in zip(names, params):
            assert rel_fro(p, want["w"][n]) < 1e-5, (tag, n)
            assert rel_fro(p.grad, want["grad_after"][n]) < 1e-6, (tag, n)
            if float(want["buf"][n].abs().max()) > 0:
                assert rel_fro(opt.state[p]["previous_grad"], want["buf"][n]) < 1e-6, (tag, n)


def test_projected_update_r50_shapes(pkg, engine):
    """update @ P at layer shapes of the R50-FPN protected set (SURVEY.md App. A),
    'backbone' scaling included, against the oracle step in fp64."""
    shapes = {"backbone.layer2.0.conv2.weight": (128, 128, 3, 3),
              "backbone.layer3.0.conv1.weight": (256, 512, 1, 1),
              "neck.fpn_convs.0.conv.weight": (256, 256, 3, 3),
              "neck.lateral_convs.0.conv.weight": (256, 256, 1, 1),
              "backbone.layer2.0.bn2.weight": (128,)}
    g = torch.Generator().manual_seed(1)
    transforms = {}
    for n, s in shapes.items():
        if len(s) == 4:
            d = s[1] * s[2] * s[3]
            transforms[n] = synth.decaying_cov(d, d, rank=17)
            ev, evec = torch.linalg.eigh(transforms[n].double())
            basis = evec[:, :d - 17]
            P = basis @ basis.t()
            if "backbone" in n:
                P = P / torch.linalg.norm(P)
            transforms[n] = P.float()
    init = {n: torch.randn(*s, generator=g) for n, s in shapes.items()}
    kw = dict(lr=0.02, momentum=0.9, weight_decay=1e-4)
    names = list(shapes)
    params = [torch.nn.Parameter(init[n].clone().cuda()) for n in names]
    opt = pkg.SGDNSCL(params, svd=True, **kw)
    opt.param_groups[0]["names"] = names
    for n, P in transforms.items():
        opt.transforms[n] = P.cuda()
    ref_p = {n: init[n].double().clone() for n in names}
    ref_t = {n: P.double() for n, P in transforms.items()}
    states = {}
    for step in range(2):
        grads = {n: torch.randn(*shapes[n], generator=g) for n in names}
        for n, p in zip(names, params):
            p.grad = grads[n].clone().cuda()
        opt.step()
        O.sgd_nscl_step(ref_p, {n: v.double() for n, v in grads.items()}, states, ref_t,
                        svd=True, **kw)
        for n, p in zip(names, params):
            assert rel_fro(p, ref_p[n]) < 1e-6, (step, n)
    # the projected update in isolation: start from W = 0 so that W_new IS the update
    # (no cancellation against fp32 rounding of W, which alone is ~1e-4 of a
    # backbone-scaled update)
    zparams = [torch.nn.Parameter(torch.zeros(shapes[n], device="cuda")) for n in names]
    zopt = pkg.SGDNSCL(zparams, svd=True, **kw)
    zopt.param_groups[0]["names"] = names
    for n, P in transforms.items():
        zopt.transforms[n] = P.cuda()
    grads = {n: torch.randn(*shapes[n], generator=g) for n in names}
    for n, p in zip(names, zparams):
        p.grad = grads[n].clone().cuda()
    zopt.step()
    zref = {n: torch.zeros(shapes[n], dtype=torch.float64) for n in names}
    O.sgd_nscl_step(zref, {n: v.double() for n, v in grads.items()}, {}, ref_t, svd=True, **kw)
    for n, p in zip(names, zparams):
        assert rel_fro(p, zref[n]) < TOL, n


@pytest.mark.parametrize("name", ["backbone.layer3.0.conv2.weight", "neck.fpn_convs.1.conv.weight"])
def test_lowrank_projection_equals_dense(pkg, engine, name):
    """step() after get_transforms uses W += s*(upd - (upd U) U^T) with U the kept-out
    eigenvectors; it must equal the dense ``update @ P`` of the reference (SGD_NSCL.py:85-95)
    with P built by the reference's own recipe (fp32 SVD, oracle), 'backbone' scale included."""
    d, cout = 1152, 256
    cov = synth.decaying_cov(d, 11, rank=23)
    g = torch.Generator().manual_seed(3)
    grad = torch.randn(cout, 128, 3, 3, generator=g)
    kw = dict(lr=0.02, momentum=0.9, weight_decay=1e-4)
    # fp64 run of the reference recipe = the truth line (SURVEY.md App. C.4); the fp32 SVD
    # the reference itself runs carries ~1e-4 of its own noise at d = 1152
    s, v = O.eigens(cov.double())
    P_ref = O.transform(s, v, name, 0.0)
    s32, v32 = O.eigens(cov)
    assert rel_fro(O.transform(s32, v32, name, 0.0), P_ref) < 3e-4
    ref = {name: torch.zeros(cout, 128, 3, 3, dtype=torch.float64)}
    O.sgd_nscl_step(ref, {name: grad.double()}, {}, {name: P_ref.double()}, svd=True, **kw)
    outs = []
    for ratio in (0.25, 0.0):                  # low-rank form, then forced dense form
        p = torch.nn.Parameter(torch.zeros(cout, 128, 3, 3, device="cuda"))
        opt = pkg.SGDNSCL([p], svd=True, **kw)
        opt.lowrank_max_ratio = ratio
        opt.param_groups[0]["names"] = [name]
        opt.get_eigens({name: cov.cuda()})
        opt.get_transforms(offset=0.0)
        assert rel_fro(opt.transforms[name], P_ref) < TOL
        p.grad = grad.clone().cuda()
        opt.step()
        used_lowrank = opt._plans[0]["t_arena"] is not None
        assert used_lowrank == (ratio > 0)
        assert rel_fro(p, ref[name]) < TOL, ratio
        outs.append(p.detach().clone())
    assert rel_fro(outs[0], outs[1]) < 2e-5


# ----------------------------------------------------------------------- prototypes
def test_prototypes_match_reference_fixture(pkg, engine, golden_dir):
    g = _load(golden_dir, "prototypes.pt")
    feats, lab = synth.proto_features()
    mp = pkg.MultiPrototypeReplay(max_prototype=10).build(feats.cuda(), lab.cuda(), range(0, 3))
    assert torch.equal(mp.tmp_label.cpu(), g["tmp_label"])
    assert [len(m) for m in mp.save_idx] == [len(m) for m in g["masks"]]
    for mine, ref in zip(mp.save_idx, g["masks"]):
        for a, b in zip(mine, ref):
            assert torch.equal(a.cpu().bool(), b)
    assert rel_fro(mp.bbox_featss, g["protos"]) < 1e-5
    # next task replays the saved masks (mask.pth) and adds one class
    feats2, lab2 = synth.proto_features(seed=1, classes=4, per_class=60, bg=20)
    feats2 = torch.cat([feats, feats2[lab2 == 3]])
    lab2 = torch.cat([lab, lab2[lab2 == 3]])
    mp2 = pkg.MultiPrototypeReplay(max_prototype=10).build(
        feats2.cuda(), lab2.cuda(), range(0, 4), saved_masks=[list(m) for m in g["masks"]])
    assert torch.equal(mp2.tmp_label.cpu(), g["tmp_label2"])
    assert rel_fro(mp2.bbox_featss, g["protos2"]) < 1e-5


@pytest.mark.parametrize("seed,classes,per_class,sub,noise,max_proto,D", [
    (3, 4, 150, 12, 0.35, 10, 1024),     # more sub-clusters than picks: the cover stops at 9
    (4, 2, 333, 3, 0.60, 10, 512),       # noisy: similarities straddle 0.6, many equal counts
    (5, 5, 41, 2, 0.35, 4, 2048),        # max_prototype = 4
    (6, 3, 700, 20, 0.45, 10, 256),      # n > 2 x 256 rows per class (multi-pass compaction)
    (7, 1, 1, 1, 0.35, 10, 64),          # a class with a single row
])
def test_prototypes_device_cover_matches_oracle(pkg, seed, classes, per_class, sub, noise,
                                                max_proto, D):
    """Density ordering, greedy cover and segment table on the device against the CPU
    restatement: same labels, same picked masks, prototypes within 1e-5; then the next
    task replays a truncated mask list (mask.pth) and continues the cover."""
    feats, lab = synth.proto_features(seed=seed, classes=classes, per_class=per_class, D=D,
                                      sub=sub, noise=noise, bg=17)
    want_p, want_l, want_m = O.build_prototypes(feats, lab, range(classes), max_proto)
    mp = pkg.MultiPrototypeReplay(max_prototype=max_proto).build(feats.cuda(), lab.cuda(),
                                                                 range(classes))
    assert torch.equal(mp.tmp_label.cpu(), want_l)
    assert [len(m) for m in mp.save_idx] == [len(m) for m in want_m]
    for mine, ref in zip(mp.save_idx, want_m):
        for a, b in zip(mine, ref):
            assert torch.equal(a.cpu().bool(), b.bool())
    assert rel_fro(mp.bbox_featss, want_p) < 1e-5
    # replay: keep only the first pick of every class, the cover continues after it
    saved = [[m.clone() for m in ms[:1]] for ms in want_m]
    want_p2, want_l2, want_m2 = O.build_prototypes(feats, lab, range(classes), max_proto,
                                                   saved_masks=[list(m) for m in saved])
    mp2 = pkg.MultiPrototypeReplay(max_prototype=max_proto).build(
        feats.cuda(), lab.cuda(), range(classes), saved_masks=[list(m) for m in saved])
    assert torch.equal(mp2.tmp_label.cpu(), want_l2)
    for mine, ref in zip(mp2.save_idx, want_m2):
        assert len(mine) == len(ref)
        for a, b in zip(mine, ref):
            assert torch.equal(a.cpu().bool(), b.bool())
    assert rel_fro(mp2.bbox_featss, want_p2) < 1e-5


def test_cosine_count_mask_vs_oracle(pkg, engine):
    """Neighbour mask / counts (:417-421): identical to the oracle except where the
    similarity is within 1e-5 of the threshold (documented near-tie rule)."""
    feats, lab = synth.proto_features(seed=4, classes=2, per_class=150, D=12544, sub=3, bg=10)
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    F = feats.cuda()
    rows = torch.nonzero(lab == 1).flatten().to(torch.int32).cuda()
    n = rows.numel()
    ws = torch.empty(lib.repre_cosine_count_workspace_bytes(n, 12544), dtype=torch.uint8,
                     device="cuda")
    mask = torch.empty(n, n, dtype=torch.uint8, device="cuda")
    cnt = torch.empty(n, dtype=torch.int32, device="cuda")
    sim = torch.empty(n, n, device="cuda")
    pkg._lib.check(lib.repre_cosine_count(ptr(F), 12544, ptr(rows), n, 0.6, ptr(mask), ptr(cnt),
                                          ptr(sim), ptr(ws), ws.numel(), _stream()), "cosine")
    s_ref, m_ref, c_ref = O.cosine_neighbour_mask(feats[lab == 1].double())
    assert rel_fro(sim, s_ref) < 1e-5
    differ = mask.cpu().bool() != m_ref
    assert bool(((s_ref - 0.6).abs()[differ] < 1e-5).all())
    assert torch.equal(cnt.cpu().long(), mask.cpu().long().sum(-1))
    if not differ.any():
        assert torch.equal(cnt.cpu().long(), c_ref)


def test_class_index_and_segment_mean_edge_cases(pkg):
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    g = torch.Generator().manual_seed(2)
    M, D, C = 1000, 256, 7
    lab = torch.randint(0, C + 2, (M,), generator=g)
    lab[lab == 3] = 0                                    # class 3 empty
    F = torch.randn(M, D, generator=g)
    counts = torch.empty(C, dtype=torch.int32, device="cuda")
    offsets = torch.empty(C + 1, dtype=torch.int32, device="cuda")
    rows = torch.empty(M, dtype=torch.int32, device="cuda")
    pkg._lib.check(lib.repre_class_index(ptr(lab.cuda()), M, C, ptr(counts), ptr(offsets),
                                         ptr(rows), _stream()), "class_index")
    off = offsets.cpu().tolist()
    for c in range(C):
        want = torch.nonzero(lab == c).flatten()
        assert counts[c].item() == want.numel()
        assert torch.equal(rows[off[c]:off[c + 1]].cpu().long(), want)      # bit-exact, stable
    out = torch.empty(C, D, device="cuda")
    mx = int(counts.max().item())
    pkg._lib.check(lib.repre_segment_mean(ptr(F.cuda()), D, ptr(offsets), ptr(rows), C, mx,
                                          ptr(out), _stream()), "segment_mean")
    for c in range(C):
        if c == 3:
            assert bool(out[c].isnan().all())            # torch.mean of an empty slice
        else:
            assert rel_fro(out[c], F[lab == c].double().mean(0)) < 1e-6


def test_replay_gather_identity_index_and_gaussian(pkg):
    g = torch.Generator().manual_seed(9)
    protos = torch.randn(37, 12544, generator=g)
    mp = pkg.MultiPrototypeReplay()
    mp.bbox_featss = protos.cuda()
    out = mp.staged()
    assert torch.equal(out.cpu(), protos)                                    # bit-exact copy
    idx = torch.randperm(37, generator=g)[:16]
    assert torch.equal(mp.staged(idx=idx.cuda()).cpu(), O.replay_gather(protos, idx))
    # extension (parity unpinned by the reference): Gaussian jitter, counter-based RNG
    sigma = torch.rand(37, 12544, generator=g)
    got = mp.staged(idx=idx.cuda(), sigma=sigma.cuda(), seed=1234)
    want = O.replay_gather_gaussian(protos, sigma, idx, 1234)
    assert float((got.cpu() - want).abs().max()) < 1e-4


def test_kmeans_assign_extension(pkg, engine):
    """Extension named by BASELINE.json (no reference counterpart, parity unpinned)."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    g = torch.Generator().manual_seed(6)
    n, k, D = 500, 12, 12544
    cent = torch.randn(k, D, generator=g)
    x = cent[torch.randint(0, k, (n,), generator=g)] + 0.5 * torch.randn(n, D, generator=g)
    ws = torch.empty(lib.repre_kmeans_assign_workspace_bytes(n, k, D), dtype=torch.uint8,
                     device="cuda")
    lab = torch.empty(n, dtype=torch.int64, device="cuda")
    # named, not temporaries: a freed temporary's memory can go to the next .cuda() copy
    # before the kernel has read it
    x_d, cent_d = x.cuda(), cent.cuda()
    pkg._lib.check(lib.repre_kmeans_assign(ptr(x_d), n, D, ptr(cent_d), k, ptr(lab), ptr(ws),
                                           ws.numel(), _stream()), "kmeans")
    want, _ = O.kmeans_assign(x.double(), cent.double())
    assert torch.equal(lab.cpu(), want)


def test_kmeans_prototypes_extension(pkg):
    """Lloyd iterations on the device (assign + segmented-mean update, an empty cluster keeps
    its centre) against the plain-torch definition; parity unpinned by the reference."""
    g = torch.Generator().manual_seed(8)
    n, k, D = 700, 9, 12544
    true = torch.randn(k - 1, D, generator=g)
    x = true[torch.randint(0, k - 1, (n,), generator=g)] + 0.6 * torch.randn(n, D, generator=g)
    init = torch.cat([x[torch.randperm(n, generator=g)[:k - 1]], 50.0 + torch.randn(1, D, generator=g)])
    cent = init.double()
    for _ in range(4):
        lab, _ = O.kmeans_assign(x.double(), cent)
        cent = O.kmeans_update(x.double(), lab, k, cent)
    want_lab, _ = O.kmeans_assign(x.double(), cent)
    got_c, got_l = pkg.kmeans_prototypes(x.cuda(), init.cuda(), iters=4)
    assert torch.equal(got_l.cpu(), want_lab)
    assert rel_fro(got_c, cent) < 1e-5
    assert torch.equal(got_c[k - 1].cpu(), init[k - 1])          # the far-away centre stayed empty


def test_head_loss_adds_replay_loss(pkg, tmp_path):
    """StandardMultiPrototypeReplayHead drop-in: artifacts in, mask.pth out,
    replay_loss_cls equal to the oracle's double-softmax CE (:497-499)."""
    feats, lab = synth.proto_features(classes=3, per_class=40, D=12544, bg=10)
    prev, cur = tmp_path / "x_1", tmp_path / "x_2"
    prev.mkdir(), cur.mkdir()
    M = feats.shape[0]
    torch.save([feats, lab, torch.ones(M), torch.zeros(M, 4), torch.zeros(M, 4),
                torch.zeros(M, 5)], str(prev / "rois_etc.pth"))

    class Head(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc = torch.nn.Linear(12544, 6)

        def forward(self, x):
            return self.fc(x), None

    torch.manual_seed(0)
    head = pkg.StandardMultiPrototypeReplayHead(
        bbox_head=Head().cuda(), previous_path=str(prev), task_id=2, task_split=[0, 3, 5],
        max_prototype=10)
    assert head.replay and os.path.exists(str(cur / "mask.pth"))
    losses = head.loss()
    protos, tmp_label, _ = O.build_prototypes(feats, lab, range(0, 3), max_proto=10)
    score = head.bbox_head.fc(protos.cuda())
    want = O.replay_loss(score.cpu(), tmp_label, 5)
    assert abs(float(losses["replay_loss_cls"]) - float(want)) < 1e-5


# ------------------------------------------------------------------ SURVEY 8(f)-3 / 8(f)-4
def test_pseudo_label_merge_matches_reference_fixture(pkg, golden_dir):
    """One kernel for the whole batch against the outputs of the reference's own
    FasterRCNNRoIReplay.loss: boxes and labels bit-exact, same order."""
    cases = _load(golden_dir, "pseudo_merge.pt")
    for case in cases:
        gt_b, gt_l, ps_b, ps_s, ps_l = synth.pseudo_label_case(case["seed"])
        cu = lambda ts: [t.cuda() for t in ts]
        got = pkg.merge_pseudo_labels(cu(gt_b), cu(gt_l), cu(ps_b), cu(ps_s), cu(ps_l))
        for mine, ref in zip(got, case["out"]):
            for a, b in zip(mine, ref):
                assert torch.equal(a.cpu(), b)


@pytest.mark.parametrize("seed,images,max_gt,max_pseudo", [(11, 8, 10, 100), (12, 3, 1, 400),
                                                          (13, 16, 30, 60)])
def test_pseudo_label_merge_matches_oracle_at_size(pkg, seed, images, max_gt, max_pseudo):
    """Reference-sized inputs (100 teacher boxes per image, test_cfg.rcnn.max_per_img) and
    beyond, against the CPU restatement; plus degenerate (zero-area, NaN) boxes."""
    gt_b, gt_l, ps_b, ps_s, ps_l = synth.pseudo_label_case(seed, images, max_gt, max_pseudo)
    ps_b[0][1, 2:] = ps_b[0][1, :2]                   # zero-area teacher box
    ps_b[0][2] = ps_b[0][1]                           # ... twice: IoU 0/0 = NaN
    ps_s[0][1:3] = 0.9
    if images > 2:
        ps_b[2][0, 0] = float("nan")
    want = O.pseudo_label_merge(gt_b, gt_l, ps_b, ps_s, ps_l)
    cu = lambda ts: [t.cuda() for t in ts]
    got = pkg.merge_pseudo_labels(cu(gt_b), cu(gt_l), cu(ps_b), cu(ps_s), cu(ps_l))
    for mine, ref in zip(got, want):
        for a, b in zip(mine, ref):
            assert torch.equal(a.cpu(), b, ) or (a.shape == b.shape and torch.equal(
                torch.nan_to_num(a.cpu(), nan=-1.0), torch.nan_to_num(b, nan=-1.0)))


def test_pseudo_label_merge_into_samples(pkg):
    """Object-level form on the InstanceData stand-in: same samples as the tensor form."""
    from types import SimpleNamespace
    from oracle.ref_loader import Instances
    gt_b, gt_l, ps_b, ps_s, ps_l = synth.pseudo_label_case(5)
    want = O.pseudo_label_merge(gt_b, gt_l, ps_b, ps_s, ps_l)
    mk = lambda: [SimpleNamespace(gt_instances=Instances(bboxes=b.cuda(), labels=l.cuda()))
                  for b, l in zip(gt_b, gt_l)]
    samples, rpn_samples = mk(), mk()
    preds = [SimpleNamespace(pred_instances=Instances(bboxes=b.cuda(), scores=s.cuda(),
                                                      labels=l.cuda()))
             for b, s, l in zip(ps_b, ps_s, ps_l)]
    pkg.merge_into_samples(preds, samples, rpn_samples)
    for s, r, w in zip(samples, rpn_samples, want):
        assert torch.equal(r.gt_instances.bboxes.cpu(), w[0])
        assert torch.equal(r.gt_instances.labels.cpu(), w[1])
        assert torch.equal(s.gt_instances.bboxes.cpu(), w[2])
        assert torch.equal(s.gt_instances.labels.cpu(), w[3])
        assert "scores" not in s.gt_instances.keys()


def test_ewc_matches_reference_fixture(pkg, golden_dir, tmp_path):
    """Importance accumulation bit-exact with the reference's calculate_save_importance,
    EWCHook loss and gradients within 1e-5, ewc_reg_terms_ewc.pth in the same format."""
    g = _load(golden_dir, "ewc.pt")
    net = synth.ToyBNNet()
    net.load_state_dict(g["state0"])
    net = net.cuda()
    reg = pkg.register_params(net)
    assert list(reg.keys()) == g["reg_names"]
    terms = None
    tf32_was = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False           # the stand-in model's own convs in fp32
    for task, state_after in ((0, None), (1, "state2")):
        if task == 1:
            cpu_state = {k: v.cuda() for k, v in g["state2"].items()}
            net.load_state_dict(cpu_state)            # the fixture's perturbed parameters
            reg = pkg.register_params(net)
        acc = pkg.EWCImportance(reg)
        net.eval()
        batches = synth.ewc_batches(task)
        for b in batches:
            for p in net.parameters():
                p.grad = None
            torch.nn.functional.cross_entropy(net(b["inputs"].cuda()),
                                              b["data_samples"].cuda()).backward()
            # the conv / BN gradients come from cuDNN here and from MKL in the fixture: feed
            # the accumulate kernel the fixture-exact gradients separately below
            acc.accumulate(len(b), len(batches))
        terms = acc.finish(terms)
        for n in reg:
            ref = g["terms"]["importance"][n][task]
            assert rel_fro(terms["importance"][n][task], ref) < 1e-4, (task, n)
            assert torch.equal(terms["task_param"][n][task].cpu(), g["terms"]["task_param"][n][task])
    torch.backends.cudnn.allow_tf32 = tf32_was
    pkg.EWCImportance.save(terms, str(tmp_path))
    back = torch.load(str(tmp_path / "ewc_reg_terms_ewc.pth"), weights_only=False)
    assert set(back) == {"importance", "task_param"} and len(back["importance"]["bn1.weight"]) == 2
    # bit-exact arithmetic of the accumulate kernel on identical gradients
    gen = torch.Generator().manual_seed(9)
    imp0 = {n: torch.rand(p.shape, generator=gen) for n, p in reg.items()}
    grads = {n: torch.randn(p.shape, generator=gen) for n, p in reg.items()}
    want = O.ewc_accumulate({n: v.clone() for n, v in imp0.items()}, grads, 2, 7)
    acc = pkg.EWCImportance(reg)
    for n, p in reg.items():
        acc.importance[n].copy_(imp0[n])
        p.grad = grads[n].cuda()
    reg["bn1.bias"].grad = None                       # a parameter without gradient is skipped
    want["bn1.bias"] = imp0["bn1.bias"]
    acc.accumulate(2, 7)
    for n in reg:
        assert torch.equal(acc.importance[n].cpu(), want[n]), n
    # the hook: reference terms, fixture parameters
    net.load_state_dict({k: v.cuda() for k, v in g["state3"].items()})
    reg = pkg.register_params(net)
    ref_terms = {k: {n: [t.cuda() for t in v] for n, v in d.items()} for k, d in g["terms"].items()}
    hook = pkg.EWCHook(module=net, reg_params=reg, ewc_reg_terms=ref_terms)
    b = synth.ewc_batches(2)[0]
    net.train()
    for p in net.parameters():
        p.grad = None
    res = hook(b["inputs"].cuda(), b["data_samples"].cuda())
    assert set(res) == {"loss_cls", "ewc_loss"}
    assert abs(float(res["ewc_loss"]) - float(g["ewc_loss"])) <= 1e-5 * float(g["ewc_loss"])
    res["ewc_loss"].backward()
    for n, ref in g["grads"].items():
        assert rel_fro(reg[n].grad, ref) < 1e-5, n
    assert reg["bn2.bias"].grad is None
    # parameters equal to the stored ones: the reference omits the key (:1070)
    same = {"importance": {n: [v[-1]] for n, v in ref_terms["importance"].items()},
            "task_param": {n: [reg[n].detach().clone().unsqueeze(0)] for n in reg}}
    net.loss = hook.ori_loss
    hook2 = pkg.EWCHook(module=net, reg_params=reg, ewc_reg_terms=same)
    assert "ewc_loss" not in hook2(b["inputs"].cuda(), b["data_samples"].cuda())


# ------------------------------------------------------------------------ SURVEY 8(f)-2
def test_roi_extract_matches_reference_fixture(pkg, golden_dir):
    g = _load(golden_dir, "roi_extract.pt")
    feats, rois, labels = synth.roi_case(g["seed"])
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=0),
                                 out_channels=feats[0].shape[1], featmap_strides=[4, 8, 16, 32])
    assert torch.equal(ext.map_roi_levels(rois.cuda(), 4).cpu(), g["levels"])
    out = ext([f.cuda() for f in feats], rois.cuda())
    assert out.shape == g["out"].shape
    assert rel_fro(out, g["out"]) < 1e-5
    assert float((out.cpu() - g["out"]).abs().max()) < 1e-4
    # rows individually (a wrong level would be hidden in the global norm)
    per = (out.cpu() - g["out"]).flatten(1).norm(dim=1) / g["out"].flatten(1).norm(dim=1).clamp(min=1e-6)
    assert float(per.max()) < 1e-4


@pytest.mark.parametrize("sampling_ratio,levels", [(0, 4), (2, 4), (0, 1)])
def test_roi_extract_and_class_sums_r50_shape(pkg, sampling_ratio, levels):
    """256 channels, 512 proposals, four levels; features and the fused per-class sums
    against the CPU restatement."""
    strides = (4, 8, 16, 32)[:levels]
    feats, rois, labels = synth.roi_case(3, batch=2, channels=256, img_h=320, img_w=416,
                                         n_rois=512, classes=19, strides=strides)
    want, lv = O.roi_extract(feats, rois, featmap_strides=strides, sampling_ratio=sampling_ratio)
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=sampling_ratio),
                                 out_channels=256, featmap_strides=list(strides))
    cf = [f.cuda() for f in feats]
    out = ext(cf, rois.cuda())
    assert rel_fro(out, want) < 1e-5
    sums, counts, flat = ext.class_sums(cf, rois.cuda(), labels.cuda(), 19, return_feats=True)
    assert torch.equal(flat, out.flatten(1))
    want_s, want_c = O.roi_class_sums(want, labels, 19)
    assert torch.equal(counts.cpu(), want_c)
    assert rel_fro(sums, want_s) < 1e-5
    sums2, counts2 = ext.class_sums(cf, rois.cuda(), labels.cuda(), 19)       # no feature matrix
    assert torch.equal(counts2, counts) and rel_fro(sums2, want_s) < 1e-5
    # coarse prototypes = sums / counts = the prototype build's class means
    fg = counts.cpu() > 0
    mp = pkg.MultiPrototypeReplay(max_prototype=1).build(flat, labels.cuda(),
                                                         [c for c in range(19) if fg[c]])
    means = (sums / counts.clamp(min=1).unsqueeze(1))[fg.to(sums.device)]
    assert rel_fro(mp.bbox_featss, means) < 1e-5


@pytest.mark.parametrize("sampling_ratio", [0, 2])
def test_roi_extract_backward_matches_torchvision_autograd(pkg, sampling_ratio):
    """Gradient w.r.t. the four feature maps against autograd through the CPU restatement
    (torchvision roi_align per level, the reference's gather / scatter)."""
    feats, rois, labels = synth.roi_case(4, batch=2, channels=32, img_h=256, img_w=320, n_rois=96)
    gen = torch.Generator().manual_seed(0)
    gout = torch.randn(96, 32, 7, 7, generator=gen)
    ref_feats = [f.clone().requires_grad_(True) for f in feats]
    want, _ = O.roi_extract(ref_feats, rois, sampling_ratio=sampling_ratio)
    want.backward(gout)
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=sampling_ratio),
                                 32, [4, 8, 16, 32])
    cf = [f.cuda().requires_grad_(True) for f in feats]
    out = ext(cf, rois.cuda())
    assert out.requires_grad and rel_fro(out, want) < 1e-5
    out.backward(gout.cuda())
    for lvl, (mine, ref) in enumerate(zip(cf, ref_feats)):
        assert rel_fro(mine.grad, ref.grad) < 1e-5, lvl
    with torch.no_grad():                                    # no-grad path unchanged
        assert not ext(cf, rois.cuda()).requires_grad


def test_roi_extract_scale_factor_uses_unscaled_levels(pkg):
    """roi_scale_factor (:96-99): the level is mapped from the unscaled RoI, the pooling uses
    the rescaled one - against the restatement with the same order of operations."""
    from torchvision.ops import roi_align
    feats, rois, labels = synth.roi_case(9, channels=8, n_rois=48)
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=0), 8,
                                 [4, 8, 16, 32])
    lv = O.map_roi_levels(rois, 4)
    scaled = ext.roi_rescale(rois, 1.7)
    want = feats[0].new_zeros(48, 8, 7, 7)
    for i in range(4):
        inds = (lv == i).nonzero().squeeze(1)
        if inds.numel():
            want[inds] = roi_align(feats[i], scaled[inds], (7, 7), 1.0 / ext.featmap_strides[i], 0, True)
    got = ext([f.cuda() for f in feats], rois.cuda(), roi_scale_factor=1.7)
    assert rel_fro(got, want) < 1e-5
    assert not torch.equal(O.map_roi_levels(scaled, 4), lv)      # the distinction matters here


def test_roi_extract_empty_and_errors(pkg):
    feats, rois, labels = synth.roi_case(1, channels=8, n_rois=4)
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=0),
                                 out_channels=8, featmap_strides=[4, 8, 16, 32])
    out = ext([f.cuda() for f in feats], rois[:0].cuda())
    assert out.shape == (0, 8, 7, 7)
    with pytest.raises(pkg._lib.NsgpError):
        ext(feats, rois)                                   # host tensors: no CPU fallback
    with pytest.raises(pkg._lib.NsgpError):
        pkg.SingleRoIExtractor(dict(type="RoIPool", output_size=7), 8, [4])


# ------------------------------------------------------------------------- bench contract
def test_bench_line_contract(tmp_path):
    """`python bench.py` prints ONE JSON line with the keys the driver reads (small run) and
    writes the outputs of its last timed step under --dump-outputs."""
    import json
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2",
                          "--warmup", "3", "--cpu-budget-s", "0.5", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
              "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "clocks",
              "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(d["roofline"])
    # frac = ISSUED tf32 MMA FLOPs / time / burst tf32 peak: a true fraction of the tensor pipe
    assert d["roofline"]["bound"] == "tensor" and 0.3 < d["roofline"]["frac"] <= 1.0
    assert d["roofline"]["algorithmic_tflops"] > d["roofline"]["achieved"] * 0.9
    for k in ("roofline_staging", "roofline_cov_pass", "roofline_projection", "roofline_repre"):
        assert k in d, k
    assert 0.0 < d["roofline_cov_pass"]["hbm"]["frac"] <= 1.0
    assert 0.0 < d["roofline_cov_pass"]["tensor"]["frac"] <= 1.0
    assert 0.0 < d["roofline_projection"]["hbm"]["frac"] <= 1.0
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(d["cpu_baseline"])
    assert d["cpu_baseline"]["kind"] == "port"
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(d["e2e"])
    assert d["e2e"]["h2d_bytes_per_step"] > 3e8 and d["e2e"]["value"] < d["value"]
    assert d["gpu_launches"] > 0 and d["config"]["config_index"] == 1
    arrays = {f[:-4]: np.load(str(dump / f)) for f in os.listdir(str(dump))}
    assert all(f.endswith(".npy") for f in os.listdir(str(dump)))
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert len([k for k in arrays if k.startswith("cov.")]) == 61
    assert len([k for k in arrays if k.startswith("param.")]) > 0
    P = d["roofline_repre"]["prototypes"]
    assert arrays["replay_input"].size == min(P * 256 * 7 * 7, 1 << 17)   # sampled above 2^17
    assert arrays["prototype_labels"].shape == (P,)
    assert all(np.isfinite(a).all() for a in arrays.values())


def test_bench_reference_arm_loads_no_product_code():
    """`bench.py --impl reference` is the CPU port only: the product package (and with it
    libnsgp_repre_b200.so) must not be imported into that process."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', "
            "'--warmup', '0', '--config', '0']; runpy.run_path(%r, run_name='__main__'); "
            "bad = [m for m in sys.modules if m.startswith('nsgp_repre_b200')]; "
            "maps = open('/proc/self/maps').read(); "
            "assert not bad and 'libnsgp_repre_b200' not in maps, bad" %
            os.path.join(root, "bench.py"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                         timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip()][-1])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port"
    assert "batch 2" in d["cpu_baseline"]["sample"]
