"""GPU parity tests at the BASELINE.json configs the round-1 suite did not reach, and of the
drop-in callers: configs[2] (10 classes x 400-800 rows), configs[3] (4-task chain of
covariance.pth / mask.pth), configs[4] (COCO 40+40, M = 8192, B = 16), full-size FULL-matrix
covariances against fp64 on the device, one key hooked at several extents, Linear d = 12544,
per-class variance, the sampled six-tensor replay, the runner drop-in and the reference's
config keys.  Bars as in test_gpu_parity.py (1e-4 relative Frobenius; masks / labels exact)."""
import json
import os
import types

import pytest
import torch

from conftest import rel_fro, GOLDEN
from oracle import restated as O
from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


def _same_masks(mine, ref):
    assert len(mine) == len(ref)
    for a, b in zip(mine, ref):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert torch.equal(x.cpu().bool(), y.bool())


# ------------------------------------------------------------------ RePRE at configs[2] / [4]
@pytest.mark.parametrize("config", [2, 4])
def test_prototypes_at_baseline_configs(pkg, config):
    """configs[2]: 10 classes x 400-800 rows (the fine-grained case: hundreds of rows per
    class, Gram tiles off the diagonal); configs[4]: COCO 40+40, M = 16*512 = 8192 RoIs,
    40 old classes."""
    import bench
    cfg = bench.CONFIGS[config]
    feats, lab = bench.synthetic_rois(cfg["batch"], 11 + config, cfg["classes"], cfg["rois"])
    if config == 4:
        assert feats.shape == (8192, 12544)
    want_p, want_l, want_m = O.build_prototypes(feats, lab, range(cfg["classes"]), 10)
    mp = pkg.MultiPrototypeReplay(10).build(feats.cuda(), lab.cuda(), range(cfg["classes"]))
    assert torch.equal(mp.tmp_label.cpu(), want_l)
    _same_masks(mp.save_idx, want_m)
    assert rel_fro(mp.bbox_featss, want_p) < 1e-5
    assert torch.equal(mp.staged().cpu(), mp.bbox_featss.cpu())


def test_prototype_build_graph_replay_tracks_the_buffers(pkg):
    """A build repeated on the same input buffers replays a CUDA graph of its launch sequence
    from the third run on: the replay must read the buffers' CURRENT content."""
    feats, lab = synth.proto_features(seed=8, classes=4, per_class=45, D=12544, bg=20)
    f_d, l_d = feats.cuda(), lab.cuda()
    mp = pkg.MultiPrototypeReplay(10)
    want_p, want_l, want_m = O.build_prototypes(feats, lab, range(4), 10)
    for run in range(4):
        mp.build(f_d, l_d, range(4))
        assert (mp._graph is not None) == (run >= 1)
        assert torch.equal(mp.tmp_label.cpu(), want_l)
        assert rel_fro(mp.bbox_featss, want_p) < 1e-5
    _same_masks(mp.save_idx, want_m)
    # new content in the same buffers (other features, other labels): the graph follows
    feats2, lab2 = synth.proto_features(seed=9, classes=4, per_class=45, D=12544, bg=20)
    f_d.copy_(feats2)
    l_d.copy_(lab2)
    want_p2, want_l2, want_m2 = O.build_prototypes(feats2, lab2, range(4), 10)
    mp.build(f_d, l_d, range(4))
    assert torch.equal(mp.tmp_label.cpu(), want_l2)
    assert rel_fro(mp.bbox_featss, want_p2) < 1e-5
    _same_masks(mp.save_idx, want_m2)
    # an empty class is reported from a replayed build too (status word of the plan)
    l_d.copy_(torch.where(lab2 == 2, torch.full_like(lab2, 4), lab2))
    with pytest.raises(IndexError):
        mp.build(f_d, l_d, range(4))


# ------------------------------------------------------------------ configs[3]: 4-task chain
def test_four_task_chain_covariance_projector_and_masks(pkg, tmp_path):
    """VOC 5+5 multi-step: three task boundaries of cal_fea_in -> save -> (next task)
    merge_previous -> get_eigens -> get_transforms, and mask.pth replayed over three tasks,
    against the oracle chain (nsrunner_roi_replay.py:746-757, 634-662;
    standard_roi_replay_head.py:404-452)."""
    torch.manual_seed(0)
    net = synth.ToyDetector()
    net_gpu = synth.ToyDetector().cuda()
    net_gpu.load_state_dict(net.state_dict())
    split = [0, 5, 10, 15, 20]
    dirs = [tmp_path / ("x_%d" % t) for t in range(1, 5)]
    for d in dirs:
        d.mkdir()
    want_cov, prev_file = None, None
    rows_f, rows_l = [], []            # rois_etc.pth content, growing task by task
    want_saved, got_saved_path = None, None
    name = "backbone.c3x3.weight"
    for t in range(1, 5):
        # ---- covariance of task t (+ the previous tasks' file), saved as covariance.pth
        batches = synth.toy_batches(seed=10 + t, n=2, B=2)
        new = O.covariances_of_model(net, batches)
        want_cov = new if want_cov is None else {k: new[k] + want_cov[k] for k in new}
        previous = torch.load(prev_file, map_location="cuda") if prev_file else None
        path = str(dirs[t - 1] / "covariance.pth")
        got = pkg.CovarianceHooks(net_gpu, add_default_ignores=False).cal_fea_in(
            [b.cuda() for b in batches], previous=previous, save_path=path)
        assert set(got) == set(want_cov)
        for k in want_cov:
            assert rel_fro(got[k], want_cov[k]) < 1e-4, (t, k)
        prev_file = path
        # ---- next task's projector from the merged file (update_optim_transforms)
        loaded = torch.load(path, map_location="cuda")
        param = torch.nn.Parameter(net_gpu.backbone.c3x3.weight.detach().clone())
        opt = pkg.SGDNSCL([param], lr=0.02, momentum=0.9, weight_decay=1e-4, svd=True)
        opt.param_groups[0]["names"] = [name]
        opt.get_eigens({name: loaded[name]})
        opt.get_transforms(offset=0.0)
        s, v = O.eigens(want_cov[name])
        assert int(opt.adaptive_threshold(opt.eigens[name]["eigen_value"]).sum()) == \
            int(O.null_mask(s, 0.0).sum())
        assert rel_fro(opt.transforms[name], O.transform(s, v, name, 0.0)) < 5e-3
        # ---- RePRE: rois_etc.pth of task t = previous rows + this task's classes
        f_new, l_new = synth.proto_features(seed=20 + t, classes=5, per_class=30 + 3 * t,
                                            D=12544, bg=6)
        l_new = torch.where(l_new < 5, l_new + split[t - 1], torch.full_like(l_new, 20))
        rows_f.append(f_new)
        rows_l.append(l_new)
        F_all, L_all = torch.cat(rows_f), torch.cat(rows_l)
        M = F_all.shape[0]
        torch.save([F_all, L_all, torch.ones(M), torch.zeros(M, 4), torch.zeros(M, 4),
                    torch.zeros(M, 5)], str(dirs[t - 1] / "rois_etc.pth"))
        if t >= 2:
            # head of task t reads x_{t-1}: prototypes of the classes < split[t-1], replaying
            # the masks the previous head wrote, and writes mask.pth into x_t
            prev_dir = dirs[t - 2]
            head = pkg.StandardMultiPrototypeReplayHead(
                bbox_head=None, previous_path=str(prev_dir), task_id=t, task_split=split,
                max_prototype=10)
            Fp, Lp = torch.cat(rows_f[:t - 1]), torch.cat(rows_l[:t - 1])
            want_p, want_l, want_saved = O.build_prototypes(
                Fp, Lp, range(split[0], split[t - 1]), 10,
                saved_masks=[list(m) for m in want_saved] if want_saved else None)
            assert torch.equal(head.tmp_label.cpu(), want_l)
            assert rel_fro(head.bbox_featss, want_p) < 1e-5
            got_saved = torch.load(str(dirs[t - 1] / "mask.pth"), map_location="cpu")
            _same_masks(got_saved, want_saved)
            assert len(got_saved) == split[t - 1]


# ------------------------------------------------------------------ full-size, full matrix
FULL = [
    # (name, Cin, H, W, k, s, p, B)  BASELINE configs[1] / [4] extents (800x1344 input)
    ("fpn_convs.0", 256, 200, 336, 3, 1, 1, 8),      # d = 2304, N = 67 200: 38 % of the FLOPs
    ("layer3.conv2", 256, 50, 84, 3, 1, 1, 8),       # d = 2304, N = 4200
    ("layer4.conv2", 512, 25, 42, 3, 1, 1, 8),       # d = 4608, N = 1050 < d
    ("layer3.0.conv2 s2", 256, 100, 168, 3, 2, 1, 8),
    ("stem", 3, 800, 1344, 7, 2, 3, 8),              # d = 147, N = 268 800
    ("lateral 1x1", 1024, 50, 84, 1, 1, 0, 8),
    ("fpn_convs.1 B=16", 256, 100, 168, 3, 1, 1, 16),
]


@pytest.mark.parametrize("name,Cin,H,W,k,s,p,B", FULL, ids=[f[0] for f in FULL])
def test_covariance_full_size_full_matrix(pkg, name, Cin, H, W, k, s, p, B):
    """Every element of the d x d result at the BASELINE extents against the oracle's
    unfold + mm evaluated in fp64 ON THE DEVICE (the CPU would need minutes)."""
    g = torch.Generator(device="cuda").manual_seed(Cin + H + B)
    x = torch.relu(torch.randn(B, Cin, H, W, device="cuda", generator=g))
    conv = torch.nn.Conv2d(Cin, 4, k, stride=s, padding=p, bias=False).cuda()
    model = torch.nn.Sequential(conv)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
    with torch.no_grad():
        model(x)
        model(x)
    hooks.remove()
    got = hooks.fea_in["0.weight"]
    want = 2.0 * O.cov_conv2d(x.double(), (k, k), (s, s), (p, p))
    assert got.shape == want.shape == (Cin * k * k, Cin * k * k)
    err = float((got.double() - want).norm() / want.norm())
    assert err < 3e-5, err
    # element-wise, relative to the matrix scale (the Frobenius norm hides single wrong tiles)
    worst = float((got.double() - want).abs().max() / want.abs().max())
    assert worst < 1e-4, worst


# ------------------------------------------------------------------ TMA-fed staging, any batch
class _FourLayouts(torch.nn.Module):
    """One forward hooks the four staging routines the TMA kernel feeds: sliding-window 3x3
    (tile-major copies + edge rows / columns / corners), flat 1x1, and the batch mean of the
    gather layouts (3x3 stride 2, 7x7 stem)."""
    def __init__(self):
        super().__init__()
        self.stem = torch.nn.Conv2d(4, 8, 7, stride=2, padding=3, bias=False)
        self.c3 = torch.nn.Conv2d(64, 8, 3, padding=1, bias=False)
        self.c1 = torch.nn.Conv2d(64, 8, 1, bias=False)
        self.s2 = torch.nn.Conv2d(64, 8, 3, stride=2, padding=1, bias=False)
        self.d2 = torch.nn.Conv2d(64, 8, 1, stride=2, bias=False)

    def forward(self, img, x):
        return self.stem(img), self.c3(x), self.c1(x), self.s2(x), self.d2(x)


@pytest.mark.parametrize("stage_sms", ["auto", 40])
@pytest.mark.parametrize("B", [1, 2, 3, 5, 8, 12, 16, 24, 32, 33])
def test_covariance_every_batch_size_through_the_staging_ring(pkg, B, stage_sms):
    """The TMA-fed staging kernel changes its box (rows per stage), ring depth and template
    instance with the batch size (1-32; 33 falls back to the register kernel); every variant
    against the oracle, pipelined over three forwards with and without a forced partition.
    Extents: image sizes that are multiples of 256 floats, W = 20 (five float4s per row, so
    chunks end inside rows and the stage-end fix-ups of the shifted copies run)."""
    g = torch.Generator(device="cuda").manual_seed(100 + B)
    img = torch.relu(torch.randn(B, 4, 32, 64, device="cuda", generator=g))
    x = torch.relu(torch.randn(B, 64, 16, 20, device="cuda", generator=g))
    model = _FourLayouts().cuda()
    old = pkg.CovarianceHooks.stage_sms
    pkg.CovarianceHooks.stage_sms = stage_sms
    try:
        hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
        with torch.no_grad():
            for _ in range(3):
                model(img, x)
        hooks.remove()
        fea = hooks.fea_in
    finally:
        pkg.CovarianceHooks.stage_sms = old
    want = {"stem": O.cov_conv2d(img.double(), (7, 7), (2, 2), (3, 3)),
            "c3": O.cov_conv2d(x.double(), (3, 3), (1, 1), (1, 1)),
            "c1": O.cov_conv2d(x.double(), (1, 1), (1, 1), (0, 0)),
            "s2": O.cov_conv2d(x.double(), (3, 3), (2, 2), (1, 1)),
            "d2": O.cov_conv2d(x.double(), (1, 1), (2, 2), (0, 0))}
    for k, w in want.items():
        got = fea[k + ".weight"].double()
        assert got.shape == w.shape
        worst = float((got - 3.0 * w).abs().max() / (3.0 * w).abs().max())
        assert worst < 1e-4, (k, B, worst)


def test_covariance_pipeline_many_forwards_fresh_inputs(pkg):
    """30 forwards with NEW activations each (new addresses: the tensor maps are re-encoded,
    the two workspace sets alternate, the contraction of forward i-1 runs beside the staging
    of forward i on a forced partition) accumulate to the sum of the oracle's per-forward
    covariances."""
    B = 8
    g = torch.Generator(device="cuda").manual_seed(7)
    model = _FourLayouts().cuda()
    old = pkg.CovarianceHooks.stage_sms
    pkg.CovarianceHooks.stage_sms = 48
    want = {}
    keep = []
    try:
        hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
        with torch.no_grad():
            for it in range(30):
                img = torch.relu(torch.randn(B, 4, 32, 64, device="cuda", generator=g))
                x = torch.relu(torch.randn(B, 64, 16, 20, device="cuda", generator=g))
                if it % 3 == 0:
                    keep.append((img, x))            # vary the allocator's reuse pattern
                model(img, x)
                for k, (t, ks, st, pd) in {"stem": (img, 7, 2, 3), "c3": (x, 3, 1, 1),
                                           "c1": (x, 1, 1, 0), "s2": (x, 3, 2, 1),
                                           "d2": (x, 1, 2, 0)}.items():
                    c = O.cov_conv2d(t.double(), (ks, ks), (st, st), (pd, pd))
                    want[k] = c if k not in want else want[k] + c
        hooks.remove()
        fea = hooks.fea_in
    finally:
        pkg.CovarianceHooks.stage_sms = old
    for k, w in want.items():
        got = fea[k + ".weight"].double()
        worst = float((got - w).abs().max() / w.abs().max())
        assert worst < 1e-4, (k, worst)


# ------------------------------------------------------------------ one key, several extents
def test_covariance_shared_module_five_levels_one_key(pkg):
    """rpn_head.rpn_conv / rpn_cls are applied to the five FPN levels: five hook calls at
    five extents accumulate into ONE key (nsrunner_roi_replay.py:893-896), the coarsest level
    smaller than 3 px (no autocorrelation form for that call)."""
    class Rpn(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.rpn_conv = torch.nn.Conv2d(16, 16, 3, padding=1)
            self.rpn_cls = torch.nn.Conv2d(16, 3, 1)

        def forward(self, feats):
            return [self.rpn_cls(torch.relu(self.rpn_conv(f))) for f in feats]

    torch.manual_seed(1)
    net = Rpn()
    gpu = Rpn().cuda()
    gpu.load_state_dict(net.state_dict())
    g = torch.Generator().manual_seed(2)
    sizes = [(40, 56), (20, 28), (10, 14), (5, 7), (2, 4)]
    batches = [[torch.relu(torch.randn(2, 16, h, w, generator=g)) for h, w in sizes]
               for _ in range(2)]
    want = O.covariances_of_model(net, batches)
    for mode in ("deferred", "grouped"):
        hooks = pkg.CovarianceHooks(gpu, add_default_ignores=False, mode=mode)
        got = hooks.cal_fea_in([[f.cuda() for f in b] for b in batches])
        assert set(got) == {"rpn_conv.weight", "rpn_cls.weight"}
        for k in want:
            assert rel_fro(got[k], want[k]) < 2e-5, (mode, k)


def test_covariance_linear_d12544(pkg):
    """roi_head.bbox_head.shared_fcs.0: d = 12 544 (629 MB of state), rank-1 per forward."""
    lin = torch.nn.Linear(12544, 8).cuda()
    model = torch.nn.Sequential(lin)
    hooks = pkg.CovarianceHooks(model, add_default_ignores=False).register()
    g = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.relu(torch.randn(512, 12544, device="cuda", generator=g)) for _ in range(2)]
    with torch.no_grad():
        for x in xs:
            model(x)
    hooks.remove()
    got = hooks.fea_in["0.weight"]
    want = sum(O.cov_linear(x.double()) for x in xs)
    assert got.shape == (12544, 12544)
    assert float((got.double() - want).norm() / want.norm()) < 1e-5


# ------------------------------------------------------------------ extensions (unpinned)
def test_class_variance_extension(pkg):
    """Per-class diagonal covariance (north_star item 3; no reference implementation - the
    in-repo definition is oracle.restated.class_variance, biased / n): the coarse segment of
    every class."""
    feats, lab = synth.proto_features(seed=4, classes=4, per_class=50, D=12544, bg=12)
    mp = pkg.MultiPrototypeReplay(10).build(feats.cuda(), lab.cuda(), range(4))
    sigma = mp.build_sigma()
    mean, var, cnt = O.class_variance(feats.double(), lab, 4)
    coarse = [i for i in range(mp.tmp_label.numel())
              if i == 0 or mp.tmp_label[i] != mp.tmp_label[i - 1]]
    assert len(coarse) == 4
    for c, i in enumerate(coarse):
        assert rel_fro(mp.bbox_featss[i], mean[c]) < 1e-5
        assert rel_fro(sigma[i] ** 2, var[c]) < 1e-4


# ------------------------------------------------------------------ a12 sampled replay
def test_sampled_six_tensor_replay_matches_reference_indexing(pkg, tmp_path):
    """StandardRoIReplayHead.loss (:53-69): randperm(M)[:64] on the default CPU generator, six
    tensors gathered; MSE between student and teacher class scores (:97)."""
    g = torch.Generator().manual_seed(9)
    M = 300
    six = [torch.randn(M, 12544, generator=g), torch.randint(0, 21, (M,), generator=g),
           torch.rand(M, generator=g), torch.randn(M, 4, generator=g),
           torch.rand(M, 4, generator=g), torch.rand(M, 5, generator=g) * 100]
    prev = tmp_path / "x_1"
    prev.mkdir()
    torch.save(six, str(prev / "rois_etc.pth"))

    class Head(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc = torch.nn.Linear(12544, 6)

        def forward(self, x):
            return self.fc(x), None

    torch.manual_seed(0)
    head = pkg.StandardRoIReplayHead(bbox_head=Head().cuda(), previous_path=str(prev))
    head.teacher_model = types.SimpleNamespace(bbox_head=Head().cuda())
    assert head.replay and head.counter == [0] * 80
    torch.manual_seed(77)
    got = head._sampled.sample()
    torch.manual_seed(77)
    mask = torch.randperm(M)[:64]                                   # :58
    for a, b in zip(got, six):
        assert torch.equal(a.cpu(), b[mask])
    torch.manual_seed(78)
    losses = head.loss()
    torch.manual_seed(78)
    mask = torch.randperm(M)[:64]
    f = six[0][mask].cuda()
    want = torch.nn.functional.mse_loss(head.bbox_head(f)[0], head.teacher_model.bbox_head(f)[0])
    assert abs(float(losses["replay_loss_cls"]) - float(want)) < 1e-6
    assert head.loss(replay=False) == {}


# ------------------------------------------------------------------ runner drop-in
class _Preproc:
    def __call__(self, data_batch, training):
        return {"inputs": data_batch["inputs"].cuda(), "data_samples": data_batch.get("samples")}


class _Detector(synth.ToyDetector):
    def __init__(self):
        super().__init__()
        self.data_preprocessor = _Preproc()

    def forward(self, inputs, data_samples=None, mode="tensor"):
        assert mode == "nullspace"
        return super().forward(inputs)


def test_runner_dropin_cal_fea_in_and_transforms(pkg, tmp_path):
    """NullSpaceRunnerMixin on a plain object: cal_fea_in (:704-763) writes covariance.pth of
    the reference content (task 2: previous file added), update_optim_transforms (:634-662)
    filters by ignore_keys and builds the projectors."""
    torch.manual_seed(0)
    model = _Detector().cuda()
    cpu = synth.ToyDetector()
    cpu.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()})
    work, prev = tmp_path / "w_2", tmp_path / "w_1"
    work.mkdir(), prev.mkdir()
    (work / "best_x.pth").write_text("ckpt")
    batches = synth.toy_batches(seed=3, n=3, B=2)
    base = O.covariances_of_model(cpu, batches)
    old = {k: torch.eye(v.shape[0]) * 0.5 for k, v in base.items()}
    torch.save(old, str(prev / "covariance.pth"))

    class Runner(pkg.NullSpaceRunnerMixin):
        pass

    r = Runner()
    r.model, r.work_dir, r.logger = model, str(work), None
    r.ignore_keys = ["fc"] + ["roi_head.bbox_head.fc_cls", "roi_head.bbox_head.fc_reg", "teacher"]
    r.task_id, r.offset, r.ckpt_keywords = 2, 0.0, "best"
    r.fea_in_load_path = str(prev / "covariance.pth")
    r.fea_in_save_path = str(work / "covariance.pth")
    loaded = []
    r.load_or_resume = lambda: loaded.append(r._load_from)
    r.cal_fea_in([{"inputs": b} for b in batches])
    assert loaded == [str(work / "best_x.pth")]
    saved = torch.load(str(work / "covariance.pth"), map_location="cpu")
    assert set(saved) == {k for k in base if not k.startswith("fc")}
    for k in saved:
        assert rel_fro(saved[k], base[k] + old[k]) < 1e-4, k
    # the hook methods keep the reference's signatures
    conv = model.backbone.c1x1
    assert r.compute_cov(conv, (torch.rand(2, 8, 6, 6, device="cuda"),), None) is None
    # projectors for the next task from that file
    named = [(n, p) for n, p in model.named_parameters() if p.dim() == 4]
    opt = pkg.SGDNSCL([p for _, p in named], lr=0.02, momentum=0.9, weight_decay=1e-4, svd=True)
    opt.param_groups[0]["names"] = [n for n, _ in named]
    r.optim_wrapper = types.SimpleNamespace(optimizer=opt)
    r.fea_in_load_path = str(work / "covariance.pth")
    r.update_optim_transforms(None)
    assert set(opt.transforms) == {n for n, _ in named}
    before = {n: t.clone() for n, t in opt.transforms.items()}
    r.update_model_transforms(None)            # same file, same offset: nothing rebuilt
    assert all(opt.transforms[n].data_ptr() == opt.transforms[n].data_ptr() and
               torch.equal(before[n], opt.transforms[n]) for n in before)
    name = "backbone.c3x3.weight"
    s, v = O.eigens(base[name] + old[name])
    assert rel_fro(opt.transforms[name], O.transform(s, v, name, 0.0)) < 5e-3


# ------------------------------------------------------------------ reference config keys
def test_reference_config_keys_feed_the_dropins(pkg, tmp_path):
    """The keys of cl_faster_rcnn_cfgs/incremental_task/cl_faster_rcnn_nsgp_repre_*.py:14-24,
    the optimizer dict of _base_/schedules/schedule_1x_sgdnscl.py:21 and runner_type of
    _base_/brnsrunetime.py:26 (tests/golden/ref_cfg_keys.json, extracted from the reference's
    files by oracle/make_cfg_fixture.py) build the drop-ins unchanged."""
    cfg = json.load(open(os.path.join(GOLDEN, "ref_cfg_keys.json")))
    reg = pkg.registry.REGISTRY
    assert cfg["runner_type"] in reg and issubclass(reg[cfg["runner_type"]],
                                                    pkg.NullSpaceRunnerMixin)
    ocfg = dict(cfg["optim_wrapper"]["optimizer"])
    lin = torch.nn.Linear(8, 8).cuda()
    opt = pkg.registry.build(ocfg, params=list(lin.parameters()))
    assert isinstance(opt, pkg.SGDNSCL)
    grp = opt.param_groups[0]
    assert (grp["lr"], grp["momentum"], grp["weight_decay"], grp["svd"]) == (0.02, 0.9, 1e-4, True)
    for fname, task in cfg["tasks"].items():
        head_cfg = dict(task["roi_head"])
        assert head_cfg["type"] in reg
        split, tid = head_cfg["task_split"], head_cfg["task_id"]
        n_old = split[tid - 1]
        # synthetic artifacts where the config's previous_path points (relative paths made
        # absolute under tmp_path; the '_N' -> '_N+1' rule of get_work_dir is kept)
        prev = tmp_path / fname / os.path.basename(head_cfg["previous_path"])
        nxt = tmp_path / fname / os.path.basename(pkg.prototypes.get_work_dir(
            head_cfg["previous_path"]))
        prev.mkdir(parents=True), nxt.mkdir(parents=True)
        feats, lab = synth.proto_features(seed=tid, classes=n_old, per_class=12, D=12544, bg=4)
        lab = torch.where(lab < n_old, lab, torch.full_like(lab, split[-1]))
        M = feats.shape[0]
        torch.save([feats, lab, torch.ones(M), torch.zeros(M, 4), torch.zeros(M, 4),
                    torch.zeros(M, 5)], str(prev / "rois_etc.pth"))
        head_cfg["previous_path"] = str(prev)
        head = pkg.registry.build(head_cfg, bbox_head=None)
        assert head.replay and head.task_id == task["task_id"]
        assert head.task_split == task["train_task_split"]
        assert head.max_proto == task["max_prototype"]
        want_p, want_l, _ = O.build_prototypes(feats, lab, range(split[0], n_old),
                                               task["max_prototype"])
        assert torch.equal(head.tmp_label.cpu(), want_l)
        assert rel_fro(head.bbox_featss, want_p) < 1e-5
        assert os.path.exists(str(nxt / "mask.pth"))
        # runner side: ignore_keys (+ the defaults of :354) select the hooked modules
        hooks = pkg.CovarianceHooks(
            torch.nn.ModuleDict({"backbone": torch.nn.Conv2d(3, 3, 1),
                                 "rpn_head": torch.nn.Conv2d(3, 3, 1),
                                 "roi_head": torch.nn.Linear(3, 3)}),
            ignore_keys=task["ignore_keys"])
        assert [n for n, _ in hooks.hooked_modules()] == ["backbone"]


# ------------------------------------------------------------------ N > 1 on NCCL
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_job_reduces_and_shards_correctly():
    """torchrun x2 over NCCL: the timed job ends with the ONE all-reduce of the flat arena; the
    finalised covariance after the reduce equals the sum of the per-rank results
    (nsrunner_roi_replay.py:746-749), the variable-length RoI gather (:73-105) and the
    class-sharded prototype build agree with the build over the gathered rows, the projector
    build is sharded by layer."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.join(root, "bench.py"),
           "--gpus", "2", "--steps", "2", "--warmup", "3", "--no-e2e", "--config", "0"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")][-1])
    assert d["n_gpus"] == 2 and len(d["per_rank_ms_per_step"]) == 2
    assert d["allreduce_check"] is True and d["allreduce_rel_err"] < 1e-6
    assert d["sharded_prototypes_check"] is True
    assert d["phase_ms"]["allreduce_buffers"] == 1          # one flat arena, one ncclAllReduce
