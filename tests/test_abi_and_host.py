"""CPU-only checks: the C-ABI library loads and exports every symbol the header
declares; host-side logic (threshold rule, path rule, registry, sharding)."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols(bringup=False):
    """Function names the header declares: the product part, or the #ifdef NSGP_BRINGUP part."""
    text = open(os.path.join(ROOT, "include", "nsgp_repre_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"#ifdef NSGP_BRINGUP(.*?)#endif", text, flags=re.S)
    assert m, "header lost its bring-up section"
    part = m.group(1) if bringup else text[:m.start()] + text[m.end():]
    return sorted(set(re.findall(r"\b((?:nsgp|repre)_[a-z0-9_]+)\s*\(", part)))


def test_library_exports_every_header_symbol():
    import subprocess
    import nsgp_repre_b200 as pkg
    syms = _header_symbols()
    assert len(syms) >= 40
    for s in syms:
        assert hasattr(pkg._lib.lib, s), "missing export %s" % s
        assert s in pkg._lib.SIGNATURES, "ctypes signature missing for %s" % s
    assert set(pkg._lib.SIGNATURES) == set(syms), "ctypes table and header disagree"
    assert pkg._lib.lib.nsgp_abi_version() == 1
    # one engine in the shipped library: no engine switch, no debug entry points, and nothing
    # exported besides the C ABI of the header
    assert not pkg._lib.HAS_BRINGUP and pkg._lib.engine() == 0
    out = subprocess.run(["nm", "-D", "--defined-only", pkg._lib.LIB_PATH], capture_output=True,
                         text=True, check=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert exported == set(syms), sorted(exported ^ set(syms))
    for s in _header_symbols(bringup=True):
        assert s in pkg._lib.BRINGUP_SIGNATURES and not hasattr(pkg._lib.lib, s)


def test_environment_switches_are_the_documented_ones():
    """Every NSGP_* variable the bring-up library (nsgp_env) or the Python layer (os.environ)
    reads is listed in DESIGN.md 6b, and every listed one is read.  NSGP_BRINGUP_LIB, which
    selects the library, is described in the text above the table."""
    pkg_dir = os.path.join(ROOT, "nsgp-repre_b200")
    read = set()
    csrc = os.path.join(pkg_dir, "csrc")
    for name in os.listdir(csrc):
        if not name.endswith((".cu", ".cuh", ".h")):
            continue
        with open(os.path.join(csrc, name), errors="replace") as f:
            read |= set(re.findall(r'\bnsgp_env\(\s*"(NSGP_[A-Z0-9_]+)"', f.read()))
    for name in os.listdir(pkg_dir):
        if name.endswith(".py"):
            with open(os.path.join(pkg_dir, name)) as f:
                read |= set(re.findall(r'\bos\.environ(?:\.get\(|\[)\s*["\'](NSGP_[A-Z0-9_]+)',
                                       f.read()))
    read.discard("NSGP_BRINGUP_LIB")
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    section = re.search(r"^## 6b\..*?(?=^## )", design, flags=re.S | re.M)
    assert section, "DESIGN.md lost section 6b"
    documented = set()
    for row in re.findall(r"^\|([^|\n]*)\|", section.group(0), flags=re.M):
        documented |= set(re.findall(r"\bNSGP_[A-Z0-9_]+", row))
    assert "NSGP_DBG_COUNTERS" in read
    assert read == documented, "read, not documented: %s; documented, not read: %s" % (
        sorted(read - documented), sorted(documented - read))


def test_layout_queries_are_host_only():
    from nsgp_repre_b200._lib import lib, CovLayout
    L = CovLayout()
    # 3x3 s1 p1, Cin=256 at 50x84: autocorrelation layout, 29 running C x C matrices
    assert lib.nsgp_cov_conv2d_layout(256, 50, 84, 3, 3, 1, 1, 1, 1, L) == 0
    assert (L.d, L.d_int, L.taps, L.kind, L.ld) == (2304, 29 * 256, 9, 1, 256)
    assert L.acc_bytes == 29 * 256 * 256 * 4
    # 3x3 s2 p1: tap-pair layout with column-shifted copies
    assert lib.nsgp_cov_conv2d_layout(256, 50, 84, 3, 3, 2, 2, 1, 1, L) == 0
    assert (L.d, L.d_int, L.taps, L.kind) == (2304, 2304, 9, 0)
    # 7x7 s2 p3 stem, Cin=3 -> explicit im2col fallback, rows padded to 8
    assert lib.nsgp_cov_conv2d_layout(3, 64, 96, 7, 7, 2, 2, 3, 3, L) == 0
    assert (L.d, L.d_int, L.taps) == (147, 152, 1)
    # 1x1 s2 downsample -> flat
    assert lib.nsgp_cov_conv2d_layout(256, 50, 84, 1, 1, 2, 2, 0, 0, L) == 0
    assert (L.d, L.d_int, L.taps) == (256, 256, 1)
    assert lib.nsgp_cov_conv2d_layout(0, 50, 84, 1, 1, 1, 1, 0, 0, L) != 0
    assert b"invalid conv geometry" in lib.nsgp_last_error()


def test_missing_gpu_fails_loudly():
    """No CPU fallback: host tensors are rejected by the product layer."""
    from nsgp_repre_b200 import CovarianceHooks, _lib
    net = torch.nn.Conv2d(8, 8, 3, padding=1)
    hooks = CovarianceHooks(torch.nn.Sequential(net))
    with pytest.raises(_lib.NsgpError):
        hooks.compute_cov(net, (torch.randn(1, 8, 5, 5),), None)


@pytest.mark.parametrize("offset", [0.0, 0.5, -0.5, 3.0])
def test_adaptive_threshold_matches_reference_fixture(golden_dir, offset):
    from nsgp_repre_b200 import SGDNSCL
    g = torch.load(os.path.join(golden_dir, "projector.pt"), weights_only=False)
    opt = SGDNSCL([torch.nn.Parameter(torch.zeros(1))], lr=0.1)
    for name, ent in g["proj"][offset].items():
        mask = opt.adaptive_threshold(ent["svals"], offset=offset)
        assert mask.dtype == torch.bool
        assert int(mask.long().argmax()) == ent["i_thres"], name
        assert bool(mask[ent["i_thres"]:].all()) and not bool(mask[:ent["i_thres"]].any())


def test_work_dir_rule():
    from nsgp_repre_b200.prototypes import get_work_dir
    assert get_work_dir("work_dirs/x_19_1_1") == "work_dirs/x_19_1_2"
    assert get_work_dir("work_dirs/coco_40_40_1") == "./"


def test_registry_names_match_reference_configs():
    from nsgp_repre_b200 import registry
    assert {"SGDNSCL", "StandardMultiPrototypeReplayHead"} <= set(registry.REGISTRY)
    opt = registry.build(dict(type="SGDNSCL", lr=0.02, momentum=0.9, weight_decay=1e-4,
                              svd=True), params=[torch.nn.Parameter(torch.zeros(2))])
    assert opt.defaults["svd"] is True and opt.defaults["momentum"] == 0.9


def test_standin_module_names_match_mmdet():
    from nsgp_repre_b200.standin import FasterRCNNStandIn
    m = FasterRCNNStandIn(with_roi=True)
    names = dict(m.named_modules())
    for n in ["backbone.conv1", "backbone.layer2.0.conv1", "backbone.layer2.0.downsample.0",
              "backbone.layer4.2.conv3", "neck.lateral_convs.3.conv", "neck.fpn_convs.0.conv",
              "rpn_head.rpn_conv", "roi_head.bbox_head.shared_fcs.0"]:
        assert n in names, n
    convs = [n for n, mod in names.items()
             if isinstance(mod, torch.nn.Conv2d) and re.match("backbone|neck", n)]
    assert len(convs) == 61          # SURVEY.md App. A: backbone + neck hooked convs
    trainable = [n for n in convs if names[n].weight.requires_grad]
    assert len(trainable) == 50      # frozen_stages=1


def test_shard_batches():
    from nsgp_repre_b200.dist import shard_batches
    got = sorted(sum((shard_batches(11, r, 4) for r in range(4)), []))
    assert got == list(range(11))


def test_roi_harvest_single_process_merge_and_reserve(tmp_path):
    """cal_rois tail (nsrunner_roi_replay.py:825-865) without a process group: reserve N
    rows per class with one permutation per class shared by the six tensors, prepend the
    previous task's rois_etc.pth, keep the list-of-6 on-disk format."""
    from nsgp_repre_b200.rois import RoIHarvest
    g = torch.Generator().manual_seed(0)
    M = 40
    cls = torch.randint(0, 4, (M,), generator=g)
    feats = torch.randn(M, 16, generator=g)
    h = RoIHarvest()
    h.add(feats[:25], cls[:25], torch.ones(25), torch.zeros(25, 4), torch.ones(25, 4),
          torch.arange(25 * 5, dtype=torch.float32).view(25, 5))
    h.add(feats[25:], cls[25:], torch.ones(15), torch.zeros(15, 4), torch.ones(15, 4),
          torch.arange(15 * 5, dtype=torch.float32).view(15, 5))
    prev = tmp_path / "t_1"
    prev.mkdir()
    old = [torch.zeros(3, 16), torch.full((3,), 9, dtype=torch.int64), torch.ones(3),
           torch.zeros(3, 4), torch.ones(3, 4), torch.zeros(3, 5)]
    torch.save(old, str(prev / "rois_etc.pth"))
    out = h.finish(work_dir=str(tmp_path), previous_dir=str(prev), task_id=2,
                   reserve_per_class=2, num_classes=4, generator=torch.Generator().manual_seed(1))
    assert len(out) == 6 and out[0].shape == (3 + 8, 16)
    assert out[1][:3].tolist() == [9, 9, 9] and out[1][3:].tolist() == [0, 0, 1, 1, 2, 2, 3, 3]
    # the same rows were picked for every tensor: features of row i belong to class out[1][i]
    for i in range(3, 11):
        src = (feats == out[0][i]).all(dim=1).nonzero().flatten()
        assert src.numel() == 1 and int(cls[src]) == int(out[1][i])
    again = torch.load(str(tmp_path / "rois_etc.pth"))
    assert isinstance(again, list) and len(again) == 6 and torch.equal(again[0], out[0])


# ----------------------------------------------------------------- SURVEY 8(f) host logic
def test_f_rows_host_logic_and_no_cpu_fallback(golden_dir):
    """CPU-side pieces of the 8(f) drop-ins: parameter registration rule (:1006-1031), the
    level-mapping rule against the reference's own map_roi_levels, and host tensors are
    rejected by every compute entry point."""
    import nsgp_repre_b200 as pkg
    from oracle import synth
    net = synth.ToyBNNet()
    reg = pkg.register_params(net)
    assert list(reg) == ["bn1.weight", "bn1.bias", "bn2.weight", "bn2.bias",
                         "layer_bn_named.weight", "layer_bn_named.bias"]
    assert pkg.register_params(net, must_names=()) .keys() == \
        {n for n, _ in net.named_parameters() if "teacher_model" not in n}
    g = torch.load(os.path.join(golden_dir, "roi_extract.pt"), weights_only=False)
    feats, rois, labels = synth.roi_case(g["seed"])
    ext = pkg.SingleRoIExtractor(dict(type="RoIAlign", output_size=7, sampling_ratio=0), 16,
                                 [4, 8, 16, 32])
    assert torch.equal(ext.map_roi_levels(rois, 4), g["levels"])
    with pytest.raises(pkg._lib.NsgpError):
        ext(feats, rois)
    gt_b, gt_l, ps_b, ps_s, ps_l = synth.pseudo_label_case(0)
    with pytest.raises(pkg._lib.NsgpError):
        pkg.merge_pseudo_labels(gt_b, gt_l, ps_b, ps_s, ps_l)
    acc = pkg.EWCImportance(reg)
    for p in reg.values():
        p.grad = torch.ones_like(p)
    with pytest.raises(pkg._lib.NsgpError):
        acc.accumulate(2, 3)
    terms = acc.finish(None)
    assert set(terms) == {"importance", "task_param"} and terms["importance"]["bn1.weight"][0].shape == (1, 8)
    hook = pkg.EWCHook(net, reg, terms)
    with pytest.raises(pkg._lib.NsgpError):
        hook.penalty()


def test_roi_selection_matches_reference_fixture(golden_dir):
    """RoIHarvest.add_selected against the reference's own get_bbox_stuff (:165-202) under the
    same global seed: same five RoIs, same order, all six tensors."""
    import collections
    import nsgp_repre_b200 as pkg
    from oracle import synth
    cases = torch.load(os.path.join(golden_dir, "roi_select.pt"), weights_only=False)
    assert [c["kind"] for c in cases] == ["few", "many", "none", "tiny"]
    for case in cases:
        args = synth.roi_select_case(case["kind"], case["seed"])
        h = pkg.RoIHarvest()
        counter = collections.defaultdict(int)
        torch.manual_seed(case["seed"])
        got = h.add_selected(*args, bg_class_id=20, counter=counter)
        assert len(got) == 6
        for a, b in zip(got, case["out"]):
            assert torch.equal(a, b), case["kind"]
        assert got[1].shape[0] == (3 if case["kind"] == "tiny" else 5)
        assert sum(counter.values()) == case["n_counted"]


def test_bench_workload_matches_survey_appendix_a():
    """bench.py's layer trace of the stand-in detector: 61 hooked backbone+neck convs, 50 of
    them trainable (protected), 1 856.5 / 118.3 algorithmic GFLOP at 800x1344 and 1 075.0 at
    608x1024 (SURVEY.md 8d, appendix A) - the workload the metric is quoted on."""
    import bench
    from nsgp_repre_b200 import standin
    layers = bench.trace_layers(800, 1344, standin)
    assert len(layers) == 61
    assert sum(1 for r in layers if r["trainable"]) == 50
    assert abs(sum(r["cov_flops"] for r in layers) / 1e9 - 1856.488) < 0.01
    assert abs(sum(r["proj_flops"] for r in layers) / 1e9 - 118.313) < 0.01
    assert sum(1 for r in layers if r["k"] == 3 and r["s"] == 1) == 17
    small = bench.trace_layers(608, 1024, standin)
    assert abs(sum(r["cov_flops"] for r in small) / 1e9 - 1074.995) < 0.01
    feats, lab = bench.synthetic_rois(8, 7)
    assert feats.shape == (4096, 12544) and int((lab < 19).sum()) == 1024


def test_auto_stage_partition_balances_with_batch_size():
    """CovarianceHooks.stage_sms = "auto": the SMs given to the staging half of the pipelined
    covariance pass grow with the batch size (more bytes to average per contracted FLOP) and
    the choice is cached per job set."""
    import types
    import bench
    from nsgp_repre_b200 import covariance as cv
    layers = bench.trace_layers(800, 1344, bench.load_standin())
    def pick(B, main_ms):
        js = cv._JobSet()
        for r in layers:
            la = types.SimpleNamespace(layout=types.SimpleNamespace(
                kind=1 if (r["k"] == 3 and r["s"] == 1 and r["Cin"] % 8 == 0) else 0))
            js.jobs.append([r["name"], (r["Cin"], r["H"], r["W"], r["k"], r["k"], r["s"], r["s"],
                                        r["p"], r["p"]), None, la, None])
            js.xs.append(object())
        hooks = cv.CovarianceHooks(torch.nn.Identity())
        hooks.main_stream_ms = main_ms
        got = hooks._auto_stage_sms(js, B)
        assert js.auto_sms == ((js.rev, B), got)
        return got
    # plain balance of the two kernels: more SMs for the staging as the batch grows
    balanced = {B: pick(B, 0.0) for B in (2, 8, 16)}
    assert 0 < balanced[2] < balanced[8] < balanced[16] <= 120
    # a caller whose own work is far more than fits a window gets the same balance point
    assert pick(8, 50.0) == balanced[8]
    # the hot path's own 0.45 ms: the partition is moved off balance so that one side ends
    # >= 0.45 ms early (measured optimum at configs[1]: 48 or 64 SMs, not 56)
    assert pick(8, 0.45) != balanced[8] and 40 <= pick(8, 0.45) <= 72
    # nothing to overlap (no sliding-window layers): no partition
    js = cv._JobSet()
    la = types.SimpleNamespace(layout=types.SimpleNamespace(kind=0))
    js.jobs.append(["a", (64, 8, 8, 1, 1, 1, 1, 0, 0), None, la, None])
    js.xs.append(object())
    assert cv.CovarianceHooks(torch.nn.Identity())._auto_stage_sms(js, 8) == 0


def test_same_input_links_pair_a_tensor_with_its_1x1_reader():
    """CovarianceHooks._same_input_links (host half of `same_input`): jobs that read the
    tensor of a 1x1 stride-1 job point at it, whatever the hook order; the reader itself and
    jobs on other tensors get -1; with two 1x1 readers the first one is the source."""
    from nsgp_repre_b200.covariance import CovarianceHooks
    s1 = (256, 200, 336, 1, 1, 1, 1, 0, 0)          # layer2.0.conv1
    s2 = (256, 200, 336, 1, 1, 2, 2, 0, 0)          # layer2.0.downsample.0
    c3 = (256, 200, 336, 3, 3, 1, 1, 1, 1)
    other = (64, 200, 336, 1, 1, 1, 1, 0, 0)
    link = CovarianceHooks._same_input_links
    assert link([s1, s2, other], ["x", "x", "y"]) == (-1, 0, -1)
    assert link([s2, c3, s1], ["x", "x", "x"]) == (2, 2, -1)          # reader hooked last
    assert link([s2, other], ["x", "x2"]) == (-1, -1)                  # no 1x1 reader of x
    assert link([s1, s1, s2], ["x", "x", "x"]) == (-1, 0, 0)
    assert link([], []) == ()
