"""The projected SGD step at every layer shape it can meet, through the sequence the runner
uses (get_eigens -> get_transforms -> SGDNSCL.step), and the other callers of the same
contraction engine with fewer than 8 operand rows.

Reference: ``oracle.restated.sgd_nscl_step`` in fp64, fed with the optimizer's own
``opt.transforms[n]``.  That keeps the step's arithmetic apart from eigensolver noise (P
against the reference recipe is pinned in test_gpu_parity.py).  The fp64 reference runs on
the device: at d = 12 544 the CPU would need minutes.

The kept-out rank r is chosen exactly through the public API: every spectrum here has its
elbow at i0 > d / 2, and ``adaptive_threshold`` reads an offset with |offset| > 1 as absolute
(i_thres = i0 + int(offset)), so ``get_transforms(offset=r - i0)`` keeps r directions out.
Layers with d <= 4 608 get a covariance with that spectrum and a dense random eigenbasis and
go through ``get_eigens`` (cuSOLVER syevd); larger ones get their eigenbasis from one
Householder reflector H = I - 2 v v^T / v^T v, exactly orthogonal and O(d^2) to build.
"""
import pytest
import torch

from oracle import restated as O

pytestmark = pytest.mark.gpu

KW = dict(lr=0.02, momentum=0.9, weight_decay=1e-4)
TOL = 1e-4          # the projected update: relative Frobenius error and worst output row
FORMS_TOL = 2e-5    # low-rank form against the dense form of the same P
STEP_TOL = 1e-6     # weights after steps from non-zero weights (as test_projected_update_r50_shapes)
ENGINE_TOL = 2e-5   # one 3xTF32 GEMM (test_contraction_gemm_3xtf32)
EIGH_MAX_D = 4608   # larger layers take the Householder eigenbasis instead of a syevd


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _randn(shape, g):
    return torch.randn(*shape, device="cuda", generator=g)


def _rel(a, b):
    a, b = a.detach().double().reshape(-1), b.detach().double().reshape(-1).to(a.device)
    return float((a - b).norm() / b.norm())


def _worst_row(a, b):
    """Largest relative error of one output row (a wrong row or ragged tile hides in the
    global norm)."""
    a = a.detach().double().reshape(a.shape[0], -1)
    b = b.detach().double().reshape(b.shape[0], -1).to(a.device)
    return float(((a - b).norm(dim=1) / b.norm(dim=1)).max())


def _spectrum(d):
    """Strictly descending: 2 -> 1 over the first d // 2 values, then a cliff to 1e-2 and a
    decay.  The elbow lands a few values past the cliff (i0 > d / 2)."""
    i = torch.arange(d, dtype=torch.float64)
    m = d // 2
    return torch.where(i < m, 2.0 - i / m, 1e-2 * torch.exp(-4.0 * (i - m) / (d - m)))


def _covariance(d, seed):
    """Q diag(_spectrum(d)) Q^T with a random orthogonal Q, in fp64 on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(d, d, dtype=torch.float64, device="cuda", generator=g))
    return (q * _spectrum(d).cuda()) @ q.t()


def _householder_eigens(d, seed):
    """opt.eigens entry with the eigenbasis H = I - 2 v v^T / v^T v."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    v = torch.randn(d, 1, dtype=torch.float64, device="cuda", generator=g)
    h = torch.eye(d, dtype=torch.float64, device="cuda")
    h.addmm_(v, v.t(), alpha=-2.0 / float(v.square().sum()))
    return {"eigen_value": _spectrum(d).float().cuda(), "eigen_vector": h.float()}


def _keep_out(opt, names, r):
    """get_transforms with the absolute offset that keeps exactly r directions of every layer
    in `names` out (their spectra must share the elbow)."""
    i0 = {int(opt.adaptive_threshold(opt.eigens[n]["eigen_value"], 0).long().argmax())
          for n in names}
    assert len(i0) == 1, i0
    i0 = i0.pop()
    assert i0 >= r + 2, (i0, r)          # |offset| <= 1 would be read as relative
    opt.get_transforms(offset=float(r - i0))
    for n in names:
        assert opt._lowrank[n][2].shape[1] == r, n


def _lowrank_operator(opt, name):
    """s (I - U U^T) in fp64: the projector the low-rank form applies.  The fp32 P that
    get_transforms builds on the device is up to ~2.5e-5 (relative Frobenius) away from it at
    d = 12 544 (measured on a B200 at a 1000 W power limit), well inside the 1e-4 projector
    bar."""
    _, _, u, s = opt._lowrank[name]
    u = u.double()
    return s * (torch.eye(u.shape[0], dtype=torch.float64, device=u.device) - u @ u.t())


def _t_arena(opt, gi=0):
    a = opt._plans[gi]["t_arena"]
    return None if a is None else a.numel()


class _Ref:
    """The fp64 oracle step, run beside an optimizer on copies of its weights."""

    def __init__(self, names, params):
        self.p = {n: p.detach().double().clone() for n, p in zip(names, params)}
        self.states = {}

    def step(self, names, grads, transforms, **kw):
        O.sgd_nscl_step({n: self.p[n] for n in names}, {n: grads[n].double() for n in names},
                        self.states, {n: P.detach().double() for n, P in transforms.items()},
                        svd=True, **kw)

    def check(self, names, params, tol=STEP_TOL, what=""):
        for n, p in zip(names, params):
            err = _rel(p, self.p[n])
            assert err < tol, (what, n, err)


# --------------------------------------------------------------- a) one layer, both forms
def _step_from_zero(pkg, name, shape, setup, ratio, grad):
    p = torch.nn.Parameter(torch.zeros(shape, device="cuda"))
    opt = pkg.SGDNSCL([p], svd=True, **KW)
    opt.lowrank_max_ratio = ratio
    opt.param_groups[0]["names"] = [name]
    setup(opt)
    p.grad = grad.clone()
    opt.step()
    return p.detach().clone(), opt


def _check_both_forms(pkg, name, shape, setup, r, seed):
    """W = 0, one step: W is the projected update.  Low-rank form, then the dense form of the
    same P (lowrank_max_ratio = 0), each against the fp64 oracle with P, the low-rank form also
    against its own operator s (I - U U^T), and the two forms against each other: within
    FORMS_TOL plus the distance between the two operators' exact results."""
    grad = _randn(shape, torch.Generator(device="cuda").manual_seed(seed))
    cout = shape[0]
    low, opt = _step_from_zero(pkg, name, shape, setup, 0.25, grad)
    assert opt._lowrank[name][2].shape[1] == r
    assert _t_arena(opt) == 3 * cout * ((r + 3) // 4 * 4)          # the low-rank form ran
    want = torch.zeros(shape, dtype=torch.float64, device="cuda")
    O.sgd_nscl_step({name: want}, {name: grad.double()}, {},
                    {name: opt.transforms[name].double()}, svd=True, **KW)
    assert _rel(low, want) < TOL, _rel(low, want)
    assert _worst_row(low, want) < TOL, _worst_row(low, want)
    want_lr = torch.zeros(shape, dtype=torch.float64, device="cuda")
    O.sgd_nscl_step({name: want_lr}, {name: grad.double()}, {},
                    {name: _lowrank_operator(opt, name)}, svd=True, **KW)
    assert _rel(low, want_lr) < FORMS_TOL, _rel(low, want_lr)
    dense, opt_d = _step_from_zero(pkg, name, shape, setup, 0.0, grad)
    assert _t_arena(opt_d) is None                                   # the dense form ran
    assert torch.equal(opt_d.transforms[name], opt.transforms[name])
    assert _rel(dense, want) < TOL, _rel(dense, want)
    assert _worst_row(dense, want) < TOL, _worst_row(dense, want)
    gap = _rel(want_lr, want)
    assert _rel(low, dense) < FORMS_TOL + gap, (_rel(low, dense), gap)


# (id, parameter name, weight shape, kept-out directions r); 'backbone' names scale P by
# 1 / ||P||_F (s in the SGD prologue, -s in the second low-rank GEMM), the others do not
LAYERS = [
    # fewer than 8 rows of U^T
    ("r1", "backbone.layer3.0.conv2.weight", (256, 128, 3, 3), 1),
    ("r3", "neck.fpn_convs.1.conv.weight", (256, 128, 3, 3), 3),
    ("r7", "backbone.layer3.0.conv2.weight", (256, 128, 3, 3), 7),
    # 8 / 16 / 32-row boxes with an out-of-bounds tail; MMA N rounded up to 16
    ("r8", "neck.fpn_convs.1.conv.weight", (256, 128, 3, 3), 8),
    ("r15", "backbone.layer3.0.conv2.weight", (256, 128, 3, 3), 15),
    ("r16", "neck.fpn_convs.1.conv.weight", (256, 128, 3, 3), 16),
    ("r17", "backbone.layer3.0.conv2.weight", (256, 128, 3, 3), 17),
    ("r33", "neck.fpn_convs.1.conv.weight", (256, 128, 3, 3), 33),
    # T spans 1, 2 or 3 column tiles; the second GEMM's K = r crosses several K blocks
    ("r127", "backbone.layer3.1.conv2.weight", (256, 256, 3, 3), 127),
    ("r128", "neck.fpn_convs.0.conv.weight", (256, 256, 3, 3), 128),
    ("r129", "backbone.layer3.1.conv2.weight", (256, 256, 3, 3), 129),
    ("r300", "neck.fpn_convs.0.conv.weight", (256, 256, 3, 3), 300),
    # rpn_cls-sized updates: fewer than 8 rows of the staged update
    ("cout3", "rpn_head.rpn_cls.weight", (3, 256, 1, 1), 40),
    ("cout7", "backbone.layer2.0.conv1.weight", (7, 256, 1, 1), 40),
    # the smallest legal box, rpn_reg, fc_cls, a ragged second row tile
    ("cout8", "neck.lateral_convs.0.conv.weight", (8, 256, 1, 1), 40),
    ("cout12", "rpn_head.rpn_reg.weight", (12, 256, 1, 1), 40),
    ("cout21", "roi_head.bbox_head.fc_cls.weight", (21, 1024), 50),
    ("cout130", "backbone.layer1.0.conv2.weight", (130, 64, 3, 3), 50),
    # layer4.x.conv3: 16 row tiles in one problem
    ("cout2048", "backbone.layer4.1.conv3.weight", (2048, 512, 1, 1), 100),
    # d % 4 != 0: padded pitch, scalar-atomic epilogue
    ("d130", "roi_head.bbox_head.fc_x.weight", (64, 130), 20),
    ("d147", "backbone.conv1.weight", (64, 3, 7, 7), 9),
    # layer4.x.conv2: 144 K blocks in one chain
    ("d4608", "backbone.layer4.1.conv2.weight", (512, 512, 3, 3), 250),
    # shared_fcs.0: dense K beyond the 160-block chain (split); P^T hi/lo is 1.26 GB
    ("d12544", "roi_head.bbox_head.shared_fcs.0.weight", (1024, 12544), 300),
]


@pytest.mark.parametrize("name,shape,r", [c[1:] for c in LAYERS], ids=[c[0] for c in LAYERS])
def test_projected_step_one_layer(pkg, name, shape, r):
    d = 1
    for s in shape[1:]:
        d *= s
    eig = {}

    def setup(opt):
        if not eig:
            if d <= EIGH_MAX_D:
                opt.get_eigens({name: _covariance(d, d + r)})
                eig.update(opt.eigens[name])
            else:
                eig.update(_householder_eigens(d, d + r))
        opt.eigens[name] = dict(eig)
        _keep_out(opt, [name], r)

    _check_both_forms(pkg, name, shape, setup, r, seed=r)


@pytest.mark.parametrize("offset", [0.0, -0.5])
def test_projected_step_fixture_layer(pkg, golden_dir, offset):
    """backbone.a.weight of tests/golden/projector.pt (d = 72, i_thres = 6 at offset 0 and 3
    at offset -0.5) with 16 output channels, through the real get_eigens / get_transforms."""
    from oracle import synth
    g = torch.load(golden_dir + "/projector.pt", map_location="cpu", weights_only=False)
    name = "backbone.a.weight"
    d, seed, rank = g["seeds"][name]
    r = g["proj"][offset][name]["i_thres"]
    cov = synth.decaying_cov(d, seed, rank=rank).cuda()

    def setup(opt):
        opt.get_eigens({name: cov})
        opt.get_transforms(offset=offset)

    _check_both_forms(pkg, name, (16, 8, 3, 3), setup, r, seed=int(100 * offset) + 7)


# ------------------------------------------------------- b) the whole protected set, one plan
def test_projected_step_whole_standin_one_plan(pkg):
    """Every trainable parameter of the R50-FPN stand-in with RPN and RoI heads in one group:
    BN and bias parameters unprojected, every conv / linear weight (rpn_cls with 3 output
    channels, shared_fcs.0 with d = 12 544 ...) projected with r spread over 1..300, the
    low-rank and the dense form in the same plan.  Three Nesterov steps with momentum and weight
    decay from random weights, every parameter against the fp64 oracle after every step: the
    dense layers with P, the low-rank layers with s (I - U U^T) (at d = 12 544 the two differ by
    more than this bar allows; test_projected_step_one_layer pins the forms against each
    other)."""
    from nsgp_repre_b200.standin import FasterRCNNStandIn
    model = FasterRCNNStandIn(with_rpn=True, with_roi=True)
    names, shapes = zip(*[(n, p.shape) for n, p in model.named_parameters() if p.requires_grad])
    del model
    g = torch.Generator(device="cuda").manual_seed(21)
    params = [torch.nn.Parameter(_randn(s, g)) for s in shapes]
    kw = dict(lr=0.02, momentum=0.9, weight_decay=1e-4, nesterov=True)
    ratio = 0.1
    opt = pkg.SGDNSCL(params, svd=True, **kw)
    opt.lowrank_max_ratio = ratio
    opt.param_groups[0]["names"] = list(names)
    spread = (1, 300, 16, 129, 3, 64, 17, 250, 7, 128, 33, 8, 200, 15, 127)
    ranks = {}
    for k, (n, p) in enumerate(zip(names, params)):
        if p.dim() not in (2, 4):
            continue
        d = p.numel() // p.shape[0]
        ranks[n] = min(spread[len(ranks) % len(spread)], d // 2 - 8)
        opt.eigens.clear()                 # get_transforms below sets this layer's offset only
        opt.eigens[n] = _householder_eigens(d, k)
        _keep_out(opt, [n], ranks[n])
    opt.eigens.clear()
    low = {n for n, r in ranks.items() if r <= ratio * (opt.transforms[n].shape[0])}
    assert "rpn_head.rpn_cls.weight" in ranks and "roi_head.bbox_head.shared_fcs.0.weight" in ranks
    assert 0 < len(low) < len(ranks), (len(low), len(ranks))
    assert any(r < 8 for r in ranks.values())
    assert len(ranks) < len(names)                    # BN and bias parameters take part too
    ref = _Ref(names, params)
    ref_t = {n: _lowrank_operator(opt, n) if n in low else opt.transforms[n] for n in ranks}
    for step in range(3):
        grads = {n: _randn(s, g) for n, s in zip(names, shapes)}
        for n, p in zip(names, params):
            p.grad = grads[n].clone()
        opt.step()
        ref.step(names, grads, ref_t, **kw)
        ref.check(names, params, what=step)
    assert set(opt._lowrank_prepared) == low
    assert set(opt._prepared) == set(ranks) - low
    assert _t_arena(opt) == 3 * sum(params[names.index(n)].shape[0] * ((ranks[n] + 3) // 4 * 4)
                                    for n in low)


# ------------------------------------------------------------- c) the plan cache across steps
# two protected layers of the same d = 576 (64 and 3 output channels): one offset gives both
# the same r
PAIR = {"backbone.layer1.0.conv2.weight": (64, 64, 3, 3), "rpn_head.cls.weight": (3, 64, 3, 3)}


def _pair(pkg, r, seed=31, **kw):
    g = torch.Generator(device="cuda").manual_seed(seed)
    names = list(PAIR)
    params = [torch.nn.Parameter(_randn(PAIR[n], g)) for n in names]
    opt = pkg.SGDNSCL(params, svd=True, **kw)
    opt.param_groups[0]["names"] = names
    opt.get_eigens({n: _covariance(576, seed + i) for i, n in enumerate(names)})
    _keep_out(opt, names, r)
    return opt, names, params, g


def _pair_arena(r):
    return 3 * (64 + 3) * ((r + 3) // 4 * 4)


@pytest.mark.parametrize("fresh", [True, False], ids=["new_grad_tensors", "same_grad_tensors"])
def test_plan_cache_gradient_tensors(pkg, fresh):
    """New gradient tensors every step, or new values written into the same tensors: then the
    tensor table is uploaded for the first two steps only (the first-step flag changes once)."""
    opt, names, params, g = _pair(pkg, 10, **KW)
    ref = _Ref(names, params)
    for step in range(4):
        grads = {n: _randn(PAIR[n], g) for n in names}
        for n, p in zip(names, params):
            if fresh or p.grad is None:
                p.grad = grads[n].clone()
            else:
                p.grad.copy_(grads[n])
        opt.step()
        ref.step(names, grads, opt.transforms, **KW)
        ref.check(names, params, what=step)
    assert _t_arena(opt) == _pair_arena(10)


def test_plan_cache_hyperparameters_change(pkg):
    opt, names, params, g = _pair(pkg, 10, **KW)
    ref = _Ref(names, params)
    for step, (lr, momentum) in enumerate([(0.02, 0.9), (0.005, 0.5), (0.1, 0.0), (0.03, 0.9)]):
        opt.param_groups[0]["lr"] = lr
        opt.param_groups[0]["momentum"] = momentum
        grads = {n: _randn(PAIR[n], g) for n in names}
        for n, p in zip(names, params):
            p.grad = grads[n].clone()
        opt.step()
        ref.step(names, grads, opt.transforms, lr=lr, momentum=momentum, weight_decay=1e-4)
        ref.check(names, params, what=step)


def test_plan_cache_transform_changed_in_place(pkg):
    """P scaled in place after a step: the next step uses the new P, through the dense form
    (the low-rank factors describe the old one)."""
    opt, names, params, g = _pair(pkg, 10, **KW)
    ref = _Ref(names, params)
    for step in range(3):
        if step == 1:
            opt.transforms[names[0]].mul_(0.5)
        grads = {n: _randn(PAIR[n], g) for n in names}
        for n, p in zip(names, params):
            p.grad = grads[n].clone()
        opt.step()
        ref.step(names, grads, opt.transforms, **KW)
        ref.check(names, params, what=step)
        if step == 0:
            assert _t_arena(opt) == _pair_arena(10)
        else:
            assert names[0] in opt._prepared
            assert _t_arena(opt) == 3 * 3 * 12            # only the 3-row layer stays low-rank


def test_plan_cache_new_task_changes_rank(pkg):
    """get_transforms again with another offset (a new task): r changes from 10 to 3, the T
    arena shrinks and the plan is rebuilt."""
    opt, names, params, g = _pair(pkg, 10, **KW)
    ref = _Ref(names, params)
    for step in range(4):
        if step == 2:
            _keep_out(opt, names, 3)
        grads = {n: _randn(PAIR[n], g) for n in names}
        for n, p in zip(names, params):
            p.grad = grads[n].clone()
        opt.step()
        ref.step(names, grads, opt.transforms, **KW)
        ref.check(names, params, what=step)
        assert _t_arena(opt) == _pair_arena(10 if step < 2 else 3)


def test_plan_cache_group_without_svd_is_not_projected(pkg):
    opt, names, params, g = _pair(pkg, 10, **KW)
    extra = "backbone.layer1.1.conv2.weight"
    q = torch.nn.Parameter(_randn((8, 64, 3, 3), g))
    opt.add_param_group({"params": [q], "names": [extra], "svd": False})
    opt.transforms[extra] = opt.transforms[names[0]].clone()
    ref = _Ref(names + [extra], params + [q])
    for step in range(3):
        grads = {n: _randn(p.shape, g) for n, p in zip(names + [extra], params + [q])}
        for n, p in zip(names + [extra], params + [q]):
            p.grad = grads[n].clone()
        opt.step()
        ref.step(names, grads, opt.transforms, **KW)
        ref.step([extra], grads, {}, **KW)
        ref.check(names + [extra], params + [q], what=step)
    assert opt._plans[1]["n_l"] == 0


# ---------------------------------------------- d) other callers with fewer than 8 operand rows
@pytest.mark.parametrize("M", [1, 3, 7])
@pytest.mark.parametrize("N", [1, 3, 7])
def test_gemm_nt_fewer_than_8_rows(pkg, M, N):
    """C += A B^T against fp64; the padding columns and the rows below C stay untouched."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    K, guard = 100, 5
    g = torch.Generator(device="cuda").manual_seed(10 * M + N)
    A, B = _randn((M, K), g), _randn((N, K), g)
    ldc = N + (-N) % 4
    C0 = _randn((M + guard, ldc), g)
    ah, al, bh, bl = (torch.empty_like(A), torch.empty_like(A), torch.empty_like(B),
                      torch.empty_like(B))
    pkg._lib.check(lib.nsgp_split_tf32(ptr(A), ptr(ah), ptr(al), A.numel(), _stream()), "split")
    pkg._lib.check(lib.nsgp_split_tf32(ptr(B), ptr(bh), ptr(bl), B.numel(), _stream()), "split")
    C = C0.clone()
    pkg._lib.check(lib.nsgp_gemm_nt(ptr(ah), ptr(al), ptr(bh), ptr(bl), M, N, K, ptr(C), ldc,
                                    _stream()), "gemm")
    want = C0[:M, :N].double() + A.double() @ B.double().t()
    assert _rel(C[:M, :N], want) < ENGINE_TOL
    assert torch.equal(C[:M, N:], C0[:M, N:])
    assert torch.equal(C[M:], C0[M:])


@pytest.mark.parametrize("k", [1, 2, 5, 7])
@pytest.mark.parametrize("n", [1, 5, 7])
def test_kmeans_assign_fewer_than_8_points_or_centres(pkg, n, k):
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    D = 1024
    g = torch.Generator().manual_seed(100 * k + n)
    cent = torch.randn(k, D, generator=g)
    x = cent[torch.randint(0, k, (n,), generator=g)] + 0.5 * torch.randn(n, D, generator=g)
    ws = torch.empty(lib.repre_kmeans_assign_workspace_bytes(n, k, D), dtype=torch.uint8,
                     device="cuda")
    lab = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    # named, not temporaries: a freed temporary's memory can go to the next .cuda() copy
    # before the kernel has read it
    x_d, cent_d = x.cuda(), cent.cuda()
    pkg._lib.check(lib.repre_kmeans_assign(ptr(x_d), n, D, ptr(cent_d), k, ptr(lab), ptr(ws),
                                           ws.numel(), _stream()), "kmeans")
    want, _ = O.kmeans_assign(x.double(), cent.double())
    assert torch.equal(lab.cpu(), want)


@pytest.mark.parametrize("n", [7, 300])
def test_kmeans_prototypes_four_centres(pkg, n):
    g = torch.Generator().manual_seed(n)
    k, D = 4, 2048
    true = 3.0 * torch.randn(k, D, generator=g)
    x = true[torch.arange(n) % k] + torch.randn(n, D, generator=g)
    init = x[:k].clone()
    cent = init.double()
    for _ in range(3):
        lab, _ = O.kmeans_assign(x.double(), cent)
        cent = O.kmeans_update(x.double(), lab, k, cent)
    want_lab, _ = O.kmeans_assign(x.double(), cent)
    got_c, got_l = pkg.kmeans_prototypes(x.cuda(), init.cuda(), iters=3)
    assert torch.equal(got_l.cpu(), want_lab)
    assert _rel(got_c, cent) < 1e-5


@pytest.mark.parametrize("n", [1, 5])
def test_cosine_count_fewer_than_8_rows(pkg, n):
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    D = 1024
    g = torch.Generator().manual_seed(n)
    F = torch.randn(n + 3, D, generator=g)
    F[n - 1] = F[0] + 0.3 * torch.randn(D, generator=g)  # n = 5: rows 0 and 4 are neighbours
    rows = torch.arange(n, dtype=torch.int32)            # rows past n are not read
    ws = torch.empty(lib.repre_cosine_count_workspace_bytes(n, D), dtype=torch.uint8,
                     device="cuda")
    mask = torch.empty(n, n, dtype=torch.uint8, device="cuda")
    cnt = torch.empty(n, dtype=torch.int32, device="cuda")
    sim = torch.empty(n, n, device="cuda")
    F_d, rows_d = F.cuda(), rows.cuda()
    pkg._lib.check(lib.repre_cosine_count(ptr(F_d), D, ptr(rows_d), n, 0.6, ptr(mask), ptr(cnt),
                                          ptr(sim), ptr(ws), ws.numel(), _stream()), "cosine")
    s_ref, m_ref, c_ref = O.cosine_neighbour_mask(F[:n].double())
    assert _rel(sim, s_ref) < 1e-5
    assert torch.equal(mask.cpu().bool(), m_ref)
    assert torch.equal(cnt.cpu().long(), c_ref)
