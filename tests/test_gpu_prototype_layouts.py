"""The RePRE prototype build at every class layout its launch chain branches on, against an fp64
restatement of standard_roi_replay_head.py:404-452 on the same inputs.

The build (``repre_class_index`` + ``repre_build_prototypes``) is a fixed chain of launches whose
sizes are decided on the device from the labels: class-index tiles of 8 192 labels (and the
two-kernel index past 256 classes), the tile pairs and K splits of the one foreground Gram, the
row offsets of ``class_first > 0``, the greedy cover, the row-split segment means.  Every case
here runs through the C ABI (a helper that mirrors ``MultiPrototypeReplay._build_device`` and
reads every output) and through ``MultiPrototypeReplay.build``.

Reference, per class: rows L2-normalised in float64, the Gram in float64 on the device, mask
``>= 0.6`` and row counts, ``oracle.restated.greedy_masks`` (stable density order, replayed
masks first), fp64 segment means.  The generator keeps every same-class similarity at least
1e-4 away from 0.6 and each case asserts it, so the masks are compared exactly:
  * sub-clusters sit on the directions of an orthonormal basis (random centres are not nearly
    orthogonal at small D);
  * a "blob" lies within 10 degrees of its direction: pairs inside >= cos 20 deg, pairs with any
    other sub-cluster <= cos 70 deg;
  * an "arc" lies on 25 positions 7 degrees apart in a plane (+-1 degree jitter): pairs are
    7k +- 2 degrees apart, never near acos(0.6) = 53.13, and the counts fall off towards the
    ends of the arc, so density ties and greedy covers vary.
Bars: masks, counts, segment tables, ``info``, labels and ``save_idx`` exact; prototypes within
1e-5 relative L2 error per row, NaN exactly where the reference has NaN.
"""
import ctypes
import math

import pytest
import torch

from oracle import restated as O

pytestmark = pytest.mark.gpu

THRESH = 0.6
MARGIN = 1e-4          # no same-class pair closer than this to the threshold (asserted)
PROTO_TOL = 1e-5       # relative L2 error of every prototype row
SENTINEL = 12345.0
BLOB_DEG = 10.0
ARC_STEP_DEG, ARC_JITTER_DEG, ARC_POSITIONS = 7.0, 1.0, 25
D_FULL = 12544


@pytest.fixture(scope="module")
def pkg():
    import nsgp_repre_b200 as pkg
    return pkg


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------ input generator
def _class_rows(n, D, gc, gd, sub_max):
    """n rows (fp64, on the device) of one class: sub-clusters of unequal sizes, blobs and arcs
    on the directions of an orthonormal basis, rows in random order and scaled by e^U(-1,1)."""
    dev = "cuda"
    if n == 0:
        return torch.zeros(0, D, dtype=torch.float64, device=dev)
    dirs = min(D, 2 * sub_max)
    q, _ = torch.linalg.qr(torch.randn(D, dirs, dtype=torch.float64, device=dev, generator=gd))
    q = q.t()
    k = int(torch.randint(1, min(sub_max, dirs, n) + 1, (1,), generator=gc))
    cuts = (torch.randperm(n - 1, generator=gc)[:k - 1] + 1).sort().values.tolist()
    parts = [b - a for a, b in zip([0] + cuts, cuts + [n])]
    out, d = [], 0
    for j, s in enumerate(parts):
        left = len(parts) - j - 1
        if s >= 4 and dirs - d - 2 >= left and bool(torch.rand(1, generator=gc) < 0.5):
            a, b = q[d], q[d + 1]
            d += 2
            m = min(ARC_POSITIONS, s)
            pos = torch.cat([torch.arange(m), torch.randint(0, m, (s - m,), generator=gc)])
            deg = pos.double() * ARC_STEP_DEG + (torch.rand(s, generator=gc, dtype=torch.float64)
                                                  * 2 - 1) * ARC_JITTER_DEG
            th = torch.deg2rad(deg).to(dev)
            out.append(th.cos()[:, None] * a + th.sin()[:, None] * b)
        else:
            c = q[d]
            d += 1
            g = torch.randn(s, D, dtype=torch.float64, device=dev, generator=gd)
            u = g - (g @ c)[:, None] * c
            u = u / u.norm(dim=1, keepdim=True)
            al = torch.deg2rad(torch.rand(s, generator=gc, dtype=torch.float64) * BLOB_DEG).to(dev)
            out.append(al.cos()[:, None] * c + al.sin()[:, None] * u)
    rows = torch.cat(out)[torch.randperm(n, generator=gc).to(dev)]
    scale = torch.exp(torch.rand(n, generator=gc, dtype=torch.float64) * 2 - 1).to(dev)
    return rows * scale[:, None]


def _layout(sizes, D=256, seed=0, order="shuffled", bg="interleaved", n_bg=23, junk=0,
            sub_max=6, mods=None):
    """Features (M, D) fp32 and labels (M,) int64 on the device: sizes[c] rows of class c,
    n_bg background rows (label len(sizes)), ``junk`` rows labelled -1 / C + 5 / C + 100.
    order: class rows sorted by class or shuffled; bg: background and junk rows interleaved,
    first or last.  mods[c]: "zero" (one all-zero row), "dups" (the second half exact copies
    and scaled copies of the first), "identical" (every row the same)."""
    gc = torch.Generator().manual_seed(1000 + seed)
    gd = torch.Generator(device="cuda").manual_seed(2000 + seed)
    C = len(sizes)
    fg, fl = [], []
    for c, n in enumerate(sizes):
        r = _class_rows(n, D, gc, gd, sub_max)
        kind = (mods or {}).get(c)
        if kind == "zero":
            r[min(3, n - 1)] = 0.0
        elif kind == "dups":
            h = n // 2
            r[h:] = r[:n - h] * torch.tensor([1.0, 3.0], dtype=torch.float64,
                                              device="cuda").repeat(n)[:n - h, None]
        elif kind == "identical":
            r[:] = r[0].clone()
        fg.append(r)
        fl.append(torch.full((n,), c, dtype=torch.int64))
    fg, fl = torch.cat(fg), torch.cat(fl)
    if order == "shuffled":
        p = torch.randperm(fl.numel(), generator=gc)
        fg, fl = fg[p.cuda()], fl[p]
    n_other = n_bg + junk
    other = torch.randn(n_other, D, dtype=torch.float64, device="cuda", generator=gd)
    ol = torch.cat([torch.full((n_bg,), C, dtype=torch.int64),
                    torch.tensor([-1, C + 5, C + 100] * junk, dtype=torch.int64)[:junk]])
    ol = ol[torch.randperm(n_other, generator=gc)]
    M = fl.numel() + n_other
    if bg == "interleaved":
        opos = torch.randperm(M, generator=gc)[:n_other].sort().values
    elif bg == "first":
        opos = torch.arange(n_other)
    else:
        opos = torch.arange(M - n_other, M)
    is_other = torch.zeros(M, dtype=torch.bool)
    is_other[opos] = True
    fpos = torch.nonzero(~is_other).flatten()
    feats = torch.empty(M, D, dtype=torch.float64, device="cuda")
    labels = torch.empty(M, dtype=torch.int64)
    feats[fpos.cuda()] = fg
    feats[opos.cuda()] = other
    labels[fpos] = fl
    labels[opos] = ol
    return feats.float().contiguous(), labels.cuda()


def _sizes_for(M, ncls, n_bg, seed):
    """ncls unequal class sizes that, with n_bg background rows, make M rows."""
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(ncls, generator=g, dtype=torch.float64) + 0.3
    n_fg = M - n_bg
    s = (w / w.sum() * n_fg).floor().long()
    s[0] += n_fg - int(s.sum())
    return s.tolist()


def _random_masks(sizes, spec, seed):
    """A mask.pth list: spec[c] = number of random masks of class c (sizes[c] entries each),
    or a list of masks as given."""
    g = torch.Generator().manual_seed(3000 + seed)
    out = []
    for c in range(max(spec) + 1):
        v = spec.get(c, 0)
        if isinstance(v, list):
            out.append(v)
        else:
            out.append([torch.rand(sizes[c], generator=g) < 0.3 for _ in range(v)])
    return out


# ------------------------------------------------------------------------------- fp64 reference
def _neighbours(F64, rows):
    """L2-normalised rows, fp64 Gram, mask >= 0.6 (NaN: not a neighbour) and row counts; asserts
    the generator's margin around the threshold."""
    fc = F64[rows]
    fn = fc / fc.norm(dim=1, keepdim=True)
    S = fn @ fn.t()
    near = int(((S - THRESH).abs() < MARGIN).sum())
    assert near == 0, "%d same-class pairs within %g of the threshold" % (near, MARGIN)
    mask = (S >= THRESH).cpu()
    return mask, mask.long().sum(1)


def _reference(feats, labels, classes, max_proto, saved=None):
    """standard_roi_replay_head.py:404-452 in fp64 over ``classes`` in order: per class the
    rows, mask, counts, picks (row within the class, -2 = replayed), segments (global rows) and
    prototypes; and the save_idx the walk leaves."""
    F64 = feats.double()
    save_idx = [list(m) for m in saved] if saved is not None else []
    out = []
    for c in classes:
        rows = torch.nonzero(labels == c).flatten()
        mask, counts = _neighbours(F64, rows)
        prev = save_idx[c] if c < len(save_idx) else None
        n_rep = min(len(prev), max_proto - 1) if prev else 0
        used, picked = O.greedy_masks(mask, counts, max_proto,
                                      list(prev) if prev is not None else None)
        n = counts.numel()
        ordered, order = counts.sort(descending=True, stable=True)
        covered = counts <= ordered[-n // 3]
        picks = []
        for k, m in enumerate(used):
            if k < n_rep:
                picks.append(-2)
            else:
                i = next(i for i in order.tolist() if not bool(covered[i]))
                assert torch.equal(mask[i], m)
                picks.append(i)
            covered = covered | m
        segs = [rows] + [rows[m.to(rows.device)] for m in used]
        out.append(dict(c=c, rows=rows.cpu(), mask=mask, counts=counts, picks=picks,
                        segs=[s.cpu() for s in segs],
                        protos=torch.stack([F64[s].mean(0) for s in segs])))
        if c < len(save_idx):
            save_idx[c] = picked
        else:
            save_idx.append(picked)
    return out, save_idx


# ------------------------------------------------------------------------------ device helper
def _device_build(pkg, feats, labels, classes, max_proto, saved=None):
    """repre_class_index + repre_build_prototypes through the C ABI for the consecutive
    ``classes``, called as MultiPrototypeReplay._build_device calls them; every output is
    returned, prefilled so that an entry the build leaves alone cannot match by chance."""
    L = pkg._lib
    lib, ptr = L.lib, L.ptr
    L.deterministic()
    M, D = feats.shape
    ncls, c0, C, mp = len(classes), classes[0], classes[-1] + 1, max_proto - 1
    assert list(classes) == list(range(c0, C))

    def full(n, fill, dtype=torch.int32):
        return torch.full((n,), fill, dtype=dtype, device="cuda")

    b = dict(cls_counts=full(C, -7), offsets=full(C + 1, -7), rows=full(M, -7),
             masks=full(M * M, 0xAB, torch.uint8), counts=full(M, -7),
             seg_off=full(ncls * (mp + 1) + 1, -7), seg_rows=full(M * (mp + 1), -7),
             seg_label=full(ncls * (mp + 1), -7), info=full(1 + ncls + ncls * mp + 2, -7),
             out=torch.full((ncls * (mp + 1), D), SENTINEL, device="cuda"))
    ws = torch.empty(int(lib.repre_build_prototypes_workspace_bytes(M, D, ncls, mp)),
                     dtype=torch.uint8, device="cuda")
    saved_dev = n_saved = lens = None
    if saved is not None:
        lists = [list(saved[c]) if c < len(saved) else [] for c in classes]
        ns = [min(len(l), mp) for l in lists]
        chunks = [m.to(torch.uint8).reshape(-1) for l, k in zip(lists, ns) for m in l[:k]]
        if chunks:
            saved_dev = torch.cat(chunks).cuda()
            n_saved = (ctypes.c_int32 * ncls)(*ns)
            lens = (ctypes.c_int32 * ncls)(*[int(l[0].numel()) if l else 0 for l in lists])
    s = _stream()
    L.check(lib.repre_class_index(ptr(labels), M, C, ptr(b["cls_counts"]), ptr(b["offsets"]),
                                  ptr(b["rows"]), s), "repre_class_index")
    L.check(lib.repre_build_prototypes(
        ptr(feats), D, M, ptr(b["rows"]), ptr(b["offsets"]), c0, ncls, THRESH, mp, ptr(saved_dev),
        n_saved, lens, ptr(b["masks"]), ptr(b["counts"]), ptr(b["seg_off"]), ptr(b["seg_rows"]),
        ptr(b["seg_label"]), ptr(b["info"]), ptr(b["out"]), ptr(ws), ws.numel(), 0, s),
        "repre_build_prototypes")
    torch.cuda.synchronize()
    return b


def _status(b, ncls, mp):
    return int(b["info"][1 + ncls + ncls * mp])


def _check_protos(got, want, what="prototypes"):
    """Relative L2 error of every row <= PROTO_TOL; NaN rows exactly where the reference's are."""
    got = got.double()
    want = want.to(got.device)
    nan_w = want.isnan().any(1)
    assert torch.equal(got.isnan().any(1), nan_w), what
    assert bool(got[nan_w].isnan().all()), what
    ok = ~nan_w
    if bool(ok.any()):
        err = (got[ok] - want[ok]).norm(dim=1) / want[ok].norm(dim=1)
        assert float(err.max()) <= PROTO_TOL, (what, float(err.max()), int(err.argmax()))


def _seg_tables(ref):
    segs = [s for r in ref for s in r["segs"]]
    off = torch.tensor([0] + [s.numel() for s in segs]).cumsum(0)
    lab = torch.tensor([r["c"] for r in ref for _ in r["segs"]], dtype=torch.int64)
    return off, torch.cat(segs), lab


def _check_device(b, ref, max_proto):
    """Every output of one device build against the reference of its classes."""
    mp, ncls = max_proto - 1, len(ref)
    info = b["info"].cpu().tolist()
    off, rows, lab = _seg_tables(ref)
    nseg = lab.numel()
    assert info[0] == nseg
    assert info[1:1 + ncls] == [len(r["picks"]) for r in ref]
    for ci, r in enumerate(ref):
        base = 1 + ncls + ci * mp
        assert info[base:base + len(r["picks"])] == r["picks"], ("picks", r["c"])
    assert info[1 + ncls + ncls * mp] == 0                                       # status
    assert info[2 + ncls + ncls * mp] == sum(r["rows"].numel() for r in ref)     # n_fg
    nn = [r["rows"].numel() for r in ref]
    masks = b["masks"][:sum(n * n for n in nn)].cpu()
    counts = b["counts"][:sum(nn)].cpu().long()
    moff = roff = 0
    for r, n in zip(ref, nn):
        assert torch.equal(masks[moff:moff + n * n].view(n, n), r["mask"].to(torch.uint8)), \
            ("mask", r["c"])
        assert torch.equal(counts[roff:roff + n], r["counts"]), ("counts", r["c"])
        moff += n * n
        roff += n
    assert torch.equal(b["seg_off"][:nseg + 1].cpu().long(), off)
    assert torch.equal(b["seg_rows"][:rows.numel()].cpu().long(), rows)
    assert torch.equal(b["seg_label"][:nseg].cpu().long(), lab)
    _check_protos(b["out"][:nseg], torch.cat([r["protos"] for r in ref]))


def _same_save_idx(mine, want):
    assert len(mine) == len(want)
    for c, (a, b) in enumerate(zip(mine, want)):
        assert len(a) == len(b), ("save_idx", c)
        for x, y in zip(a, b):
            assert torch.equal(x.cpu().bool(), y.cpu().bool()), ("save_idx", c)


def _check_product(mp, ref, save_ref):
    _, _, lab = _seg_tables(ref)
    assert torch.equal(mp.tmp_label.cpu(), lab)
    _check_protos(mp.bbox_featss, torch.cat([r["protos"] for r in ref]), "product prototypes")
    _same_save_idx(mp.save_idx, save_ref)


def _runs(classes):
    """Runs of consecutive classes, in order."""
    runs = [[classes[0]]]
    for c in classes[1:]:
        if c == runs[-1][-1] + 1:
            runs[-1].append(c)
        else:
            runs.append([c])
    return runs


# ----------------------------------------------------------------------------------- the cases
_SMALL = [150, 40, 7, 129]
CASES = {
    # 1. tile edges of the foreground Gram (128-row tiles)
    "tiles_127_1": dict(sizes=[127, 1]),
    "tiles_128": dict(sizes=[128]),
    "tiles_129": dict(sizes=[129]),
    "tiles_128_128": dict(sizes=[128, 128]),
    "tiles_127_2_127": dict(sizes=[127, 2, 127]),
    "tiles_255_257": dict(sizes=[255, 257]),
    "tiles_130_singletons": dict(sizes=[1] * 130),
    "tiles_600_3_3": dict(sizes=[600, 3, 3]),
    "tiles_40_D12544": dict(sizes=[40], D=D_FULL),
    # 2. label forms; junk labels -1, C + 5, C + 100
    "labels_sorted_bg_interleaved": dict(sizes=[37, 90, 61, 5], order="sorted", junk=9),
    "labels_sorted_bg_first": dict(sizes=[37, 90, 61, 5], order="sorted", bg="first", junk=9),
    "labels_shuffled_bg_first": dict(sizes=[37, 90, 61, 5], bg="first", junk=9),
    "labels_shuffled_bg_last": dict(sizes=[37, 90, 61, 5], bg="last", junk=9),
    "labels_rows_below_first": dict(sizes=[50, 70, 40, 30], classes=[2, 3], junk=9),
    # 3. class_first > 0 and non-consecutive class lists
    "first5_range_5_12": dict(sizes=[30, 3, 50, 7, 44, 25, 140, 9, 60, 33, 81, 2],
                              classes=list(range(5, 12))),
    "noncons_0_1_2_5_6_9": dict(sizes=[30, 41, 12, 25, 60, 33, 70, 8, 15, 52],
                                classes=[0, 1, 2, 5, 6, 9]),
    "noncons_1_3_5": dict(sizes=[30, 41, 12, 25, 60, 33], classes=[1, 3, 5]),
    "noncons_0_2_4": dict(sizes=[30, 41, 12, 25, 60, 33], classes=[0, 2, 4]),
    # 4. M across the 8 192-label tiles of the class index
    "rows_8191": dict(M=8191, ncls=40),
    "rows_8192": dict(M=8192, ncls=40),
    "rows_8193": dict(M=8193, ncls=40),
    "rows_16385": dict(M=16385, ncls=40),
    "rows_20000_D12544": dict(M=20000, ncls=40, D=D_FULL),
    # 5. class index past its single-launch limit (256 classes) and at it
    "classes_300": dict(tiny=300),
    "classes_256": dict(tiny=256),
    # 6. D: K tail not a multiple of 32, fewer than 4 K blocks, one and two 64-block chains
    "D4": dict(sizes=_SMALL, D=4),
    "D36": dict(sizes=_SMALL, D=36),
    "D100": dict(sizes=_SMALL, D=100),
    "D2048": dict(sizes=_SMALL, D=2048),
    "D2080": dict(sizes=_SMALL, D=2080),
    "D12544": dict(sizes=_SMALL, D=D_FULL),
    # 7. max_prototype: coarse only, one pick, the default, more picks than sub-clusters
    "maxproto_1": dict(sizes=[200, 90, 33], max_proto=1),
    "maxproto_2": dict(sizes=[200, 90, 33], max_proto=2),
    "maxproto_10": dict(sizes=[200, 90, 33], max_proto=10),
    "maxproto_20": dict(sizes=[200, 90, 33], max_proto=20, sub_max=3),
    # 8. an all-zero row, exact and scaled duplicates, a class of identical rows, 2-row classes
    "degenerate": dict(sizes=[60, 45, 30, 2, 50, 2],
                       mods={0: "zero", 1: "dups", 2: "identical", 4: "dups"}),
    # 9. replayed mask.pth: n_saved = max_picks (and more), masks for some classes only, an
    #    all-False mask (empty segment), replay with class_first > 0 (the entries below it have
    #    the wrong length: reading them would fail the build)
    "replay_full": dict(sizes=[80, 60, 45], saved={0: 9, 1: 11, 2: 2}),
    "replay_some": dict(sizes=[70, 50, 90, 40], saved={0: 0, 1: 1, 2: 0}),
    "replay_all_false": dict(sizes=[70, 50, 90], saved={1: "all_false", 2: 1}),
    "replay_first3": dict(sizes=[20, 30, 25, 60, 45, 70], classes=[3, 4, 5],
                          saved={0: "wrong", 1: "wrong", 2: "wrong", 3: 2, 5: 4}),
}
DET_CASES = [k for k in CASES if k.startswith(("tiles_", "rows_", "D"))]


def _make(name):
    kw = dict(CASES[name])
    seed = sorted(CASES).index(name)
    max_proto = kw.pop("max_proto", 10)
    saved_spec = kw.pop("saved", None)
    classes = kw.pop("classes", None)
    if "M" in kw:
        sizes = _sizes_for(kw.pop("M"), kw.pop("ncls"), 23, seed)
    elif "tiny" in kw:
        g = torch.Generator().manual_seed(seed)
        sizes = torch.randint(3, 10, (kw.pop("tiny"),), generator=g).tolist()
    else:
        sizes = kw.pop("sizes")
    feats, labels = _layout(sizes, seed=seed, **kw)
    if classes is None:
        classes = list(range(len(sizes)))
    saved = None
    if saved_spec is not None:
        spec = {}
        for c, v in saved_spec.items():
            if v == "all_false":
                spec[c] = [torch.zeros(sizes[c], dtype=torch.bool),
                           torch.rand(sizes[c]) < 0.3]
            elif v == "wrong":
                spec[c] = [torch.ones(sizes[c] + 1, dtype=torch.bool)]
            else:
                spec[c] = v
        saved = _random_masks(sizes, spec, seed)
    return feats, labels, classes, max_proto, saved


@pytest.mark.parametrize("name", list(CASES))
def test_build_matches_fp64_reference(pkg, name):
    """Every output of the device build of each consecutive run of the class list, and the
    product's labels, save_idx and prototypes, against the fp64 restatement."""
    feats, labels, classes, max_proto, saved = _make(name)
    ref, save_ref = _reference(feats, labels, classes, max_proto, saved)
    by_class = {r["c"]: r for r in ref}
    for run in _runs(classes):
        b = _device_build(pkg, feats, labels, run, max_proto, saved)
        _check_device(b, [by_class[c] for c in run], max_proto)
        del b
    mp = pkg.MultiPrototypeReplay(max_proto).build(feats, labels, classes, saved)
    _check_product(mp, ref, save_ref)
    if len(_runs(classes)) > 1:
        # the mask.pth rule of the reference itself (:425-452), on the same list
        _, _, want = O.build_prototypes(feats.cpu(), labels.cpu(), classes, max_proto, saved)
        _same_save_idx(mp.save_idx, want)


@pytest.mark.parametrize("sizes,classes,empty", [
    ([0, 30, 40], [0, 1, 2], 0),
    ([30, 0, 40], [0, 1, 2], 1),
    ([30, 40, 0], [0, 1, 2], 2),
    ([20, 30, 25, 0, 40], [2, 3, 4], 3),
], ids=["first", "middle", "last", "class_first_2"])
def test_empty_class_raises_index_error(pkg, sizes, classes, empty):
    """An old class without rows: status 1 from the device, IndexError naming the class from
    the product (the reference dies in sim_sum[-0 // 3] at :422)."""
    feats, labels = _layout(sizes, seed=50 + empty)
    b = _device_build(pkg, feats, labels, classes, 10)
    assert _status(b, len(classes), 9) == 1
    with pytest.raises(IndexError, match="class %d has no stored" % empty):
        pkg.MultiPrototypeReplay(10).build(feats, labels, classes)


def test_replayed_mask_of_wrong_length_raises(pkg):
    sizes = [30, 40]
    feats, labels = _layout(sizes, seed=60)
    saved = [[torch.rand(30) < 0.5], [torch.ones(41, dtype=torch.bool)]]
    b = _device_build(pkg, feats, labels, [0, 1], 10, saved)
    assert _status(b, 2, 9) == 2
    with pytest.raises(IndexError, match="replayed mask"):
        pkg.MultiPrototypeReplay(10).build(feats, labels, [0, 1], saved)


@pytest.mark.parametrize("name", DET_CASES)
def test_deterministic_build_is_bitwise_and_matches_default(pkg, name):
    """Under torch.use_deterministic_algorithms(True) two builds are bitwise equal, match the
    fp64 reference, and give the masks, counts, segments and labels of the default mode."""
    feats, labels, classes, max_proto, saved = _make(name)
    ref, _ = _reference(feats, labels, classes, max_proto, saved)
    default = _device_build(pkg, feats, labels, classes, max_proto, saved)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        first = _device_build(pkg, feats, labels, classes, max_proto, saved)
        second = _device_build(pkg, feats, labels, classes, max_proto, saved)
    finally:
        torch.use_deterministic_algorithms(was)
        pkg._lib.deterministic()
    _check_device(first, ref, max_proto)
    for k, v in first.items():
        a, b2 = v.view(torch.int32) if v.dtype == torch.float32 else v, second[k]
        b2 = b2.view(torch.int32) if b2.dtype == torch.float32 else b2
        assert torch.equal(a, b2), k
    for k in ("masks", "counts", "seg_off", "seg_rows", "seg_label", "info"):
        assert torch.equal(first[k], default[k]), k


def test_graph_replay_past_one_class_index_tile(pkg):
    """M = 9 000 (two class-index tiles): from the third build on the same buffers the launch
    sequence is a replayed CUDA graph, which must follow content changed in place."""
    sizes = _sizes_for(9000, 40, 23, 70)
    feats, labels = _layout(sizes, seed=70)
    ref, save_ref = _reference(feats, labels, range(40), 10)
    mp = pkg.MultiPrototypeReplay(10)
    for run in range(3):
        mp.build(feats, labels, range(40))
        assert (mp._graph is not None) == (run >= 1)
        _check_product(mp, ref, save_ref)
    feats2, labels2 = _layout(sizes, seed=71)
    feats.copy_(feats2)
    labels.copy_(labels2)
    ref2, save_ref2 = _reference(feats, labels, range(40), 10)
    mp.build(feats, labels, range(40))
    _check_product(mp, ref2, save_ref2)


# ----------------------------------------------------------- C-ABI entries without a caller
@pytest.mark.parametrize("D", [100, D_FULL])
def test_cosine_count_batched_against_fp64(pkg, D):
    """repre_cosine_count_batched over classes of 0, 1, 7, 8, 129 and 300 rows: classes of
    fewer than 8 rows are contracted as 8 rows reading into the next class."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    sizes = [0, 1, 7, 8, 129, 300]
    feats, labels = _layout(sizes, D=D, seed=80)
    F64 = feats.double()
    per = [torch.nonzero(labels == c).flatten() for c in range(len(sizes))]
    rows = torch.cat(per).to(torch.int32)
    sz = (ctypes.c_int32 * len(sizes))(*sizes)
    ws = torch.empty(int(lib.repre_cosine_count_batched_workspace_bytes(sz, len(sizes), D)),
                     dtype=torch.uint8, device="cuda")
    mask = torch.full((sum(n * n for n in sizes),), 0xAB, dtype=torch.uint8, device="cuda")
    counts = torch.full((sum(sizes),), -7, dtype=torch.int32, device="cuda")
    pkg._lib.check(lib.repre_cosine_count_batched(ptr(feats), D, ptr(rows), sz, len(sizes),
                                                  THRESH, ptr(mask), ptr(counts), ptr(ws),
                                                  ws.numel(), _stream()), "cosine_count_batched")
    mask, counts = mask.cpu(), counts.cpu().long()
    moff = roff = 0
    for c, n in enumerate(sizes):
        if n:
            want_m, want_c = _neighbours(F64, per[c])
            assert torch.equal(mask[moff:moff + n * n].view(n, n), want_m.to(torch.uint8)), c
            assert torch.equal(counts[roff:roff + n], want_c), c
        moff += n * n
        roff += n


@pytest.mark.parametrize("replay", [False, True], ids=["fresh", "replayed"])
def test_greedy_segments_on_reference_masks(pkg, replay):
    """repre_greedy_segments fed the reference's masks and counts (so it is checked apart from
    the Gram): segment tables and info exact; replayed device masks include n_saved =
    max_picks and an all-False mask."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    sizes = [1, 2, 40, 129, 300, 7, 64]
    ncls, mp = len(sizes), 9
    feats, labels = _layout(sizes, seed=90)
    saved = None
    if replay:
        saved = _random_masks(sizes, {0: 0, 1: 1, 2: [torch.zeros(40, dtype=torch.bool)],
                                      3: 9, 4: 3, 6: 12}, 90)
    ref, _ = _reference(feats, labels, range(ncls), mp + 1, saved)
    masks = torch.cat([r["mask"].reshape(-1) for r in ref]).to(torch.uint8).cuda()
    counts = torch.cat([r["counts"] for r in ref]).to(torch.int32).cuda()
    rows_sel = torch.cat([r["rows"] for r in ref]).to(torch.int32).cuda()
    sz = (ctypes.c_int32 * ncls)(*sizes)
    ids = (ctypes.c_int32 * ncls)(*range(ncls))
    saved_dev = n_saved = None
    if replay:
        ns = [min(len(saved[c]), mp) if c < len(saved) else 0 for c in range(ncls)]
        saved_dev = torch.cat([m.to(torch.uint8) for c in range(len(saved))
                               for m in saved[c][:ns[c]]]).cuda()
        n_saved = (ctypes.c_int32 * ncls)(*ns)
    ws = torch.empty(int(lib.repre_greedy_segments_workspace_bytes(sz, ncls, mp)),
                     dtype=torch.uint8, device="cuda")

    def full(n):
        return torch.full((n,), -7, dtype=torch.int32, device="cuda")

    seg_off, seg_rows = full(ncls * (mp + 1) + 1), full(sum(sizes) * (mp + 1))
    seg_label, info = full(ncls * (mp + 1)), full(ncls * (mp + 1) + 1)
    pkg._lib.check(lib.repre_greedy_segments(
        ptr(masks), ptr(counts), ptr(rows_sel), sz, ids, ncls, mp, ptr(saved_dev), n_saved,
        ptr(seg_off), ptr(seg_rows), ptr(seg_label), ptr(info), ptr(ws), ws.numel(), _stream()),
        "greedy_segments")
    off, rows, lab = _seg_tables(ref)
    nseg = lab.numel()
    h = info.cpu().tolist()
    assert h[0] == nseg
    assert h[1:1 + ncls] == [len(r["picks"]) for r in ref]
    for ci, r in enumerate(ref):
        base = 1 + ncls + ci * mp
        assert h[base:base + len(r["picks"])] == r["picks"], ci
    assert torch.equal(seg_off[:nseg + 1].cpu().long(), off)
    assert torch.equal(seg_rows[:rows.numel()].cpu().long(), rows)
    assert torch.equal(seg_label[:nseg].cpu().long(), lab)


@pytest.mark.parametrize("det", [False, True], ids=["row_splits", "deterministic"])
def test_segment_mean_dev_writes_the_live_segments_only(pkg, det):
    """repre_segment_mean_dev with the live count (5) below max_segments (9): fp64 means of the
    live segments (an empty one is NaN), the rows past the live count keep their content.  Few
    long segments take the row-split path (partial means added into zeroed rows)."""
    lib, ptr = pkg._lib.lib, pkg._lib.ptr
    g = torch.Generator(device="cuda").manual_seed(5)
    M, D, max_seg = 3000, 256, 9
    F = torch.randn(M, D, device="cuda", generator=g)
    lens = [2000, 0, 1, 37, 500]
    off = torch.tensor([0] + lens).cumsum(0).tolist()
    off = torch.tensor(off + [10 ** 9] * (max_seg - len(lens)), dtype=torch.int32, device="cuda")
    rows = torch.randint(0, M, (sum(lens),), device="cuda", generator=g, dtype=torch.int32)
    out = torch.full((max_seg, D), SENTINEL, device="cuda")
    nseg = torch.tensor([len(lens)], dtype=torch.int32, device="cuda")
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(det)
    try:
        pkg._lib.deterministic()
        pkg._lib.check(lib.repre_segment_mean_dev(ptr(F), D, ptr(off), ptr(rows), max_seg,
                                                  ptr(nseg), max(lens), ptr(out), _stream()),
                       "segment_mean_dev")
        torch.cuda.synchronize()
    finally:
        torch.use_deterministic_algorithms(was)
        pkg._lib.deterministic()
    F64, o = F.double(), off.tolist()
    want = torch.stack([F64[rows[o[s]:o[s + 1]].long()].mean(0) for s in range(len(lens))])
    _check_protos(out[:len(lens)], want, "segment means")
    assert bool((out[len(lens):] == SENTINEL).all())
