"""Cost of torch.use_deterministic_algorithms(True) on the hot path at configs[1] (B = 8,
800x1344): the bench.py step (RePRE build + covariance pass + SGDNSCL.step) and its three
phases alone, with the switch off and on, alternating in one process, plus the partial-tile
slot bytes one pass / one step writes in deterministic mode.
usage: bench_deterministic.py [rounds] [steps]   (prints one JSON line)"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
import torch

import bench
import nsgp_repre_b200 as pkg
from nsgp_repre_b200 import standin

SLOT_BYTES = 128 * 128 * 4


def gpu_info():
    q = "--query-gpu=name,power.limit"
    try:
        out = subprocess.run(["nvidia-smi", q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    cfg = bench.CONFIGS[1]
    B, H, W, C_OLD = cfg["batch"], cfg["height"], cfg["width"], cfg["classes"]
    dev = torch.device("cuda", 0)
    torch.manual_seed(1234)
    model = standin.FasterRCNNStandIn(with_rpn=False, with_roi=False).to(dev).eval()
    layers = bench.trace_layers(H, W, standin)
    modules = dict(model.named_modules())
    images = bench.synthetic_images(B, H, W, 0).to(dev)
    feats_h, labels_h = bench.synthetic_rois(B, 7, C_OLD, cfg["rois"])
    feats, labels = feats_h.to(dev), labels_h.to(dev)
    inputs, names = {}, {m: n for n, m in model.named_modules()}
    cap = [m.register_forward_hook(lambda m, i, o: inputs.__setitem__(names[m], i[0].detach()
                                                                       .contiguous()))
           for m in model.modules() if isinstance(m, torch.nn.Conv2d)]
    with torch.no_grad():
        model(images)
    for h in cap:
        h.remove()
    hooks = pkg.CovarianceHooks(model, ignore_keys=bench.IGNORE_KEYS)
    hooks._plan_arena()
    hooked = [(r["name"], modules[r["name"]]) for r in layers]

    def cov_pass():
        for n, m in hooked:
            hooks.compute_cov(m, (inputs[n],), None)
        hooks.flush()

    cov_pass()
    fea = hooks.fea_in
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    opt = pkg.SGDNSCL([p for _, p in named], lr=0.02, momentum=0.9, weight_decay=1e-4, svd=True)
    opt.param_groups[0]["names"] = [n for n, _ in named]
    opt.get_eigens(fea)
    opt.get_transforms(offset=0.0)
    del fea
    hooks.reset()
    g = torch.Generator(device=dev).manual_seed(1)
    for n, p in named:
        p.grad = torch.randn(p.shape, device=dev, generator=g)
    proto = pkg.MultiPrototypeReplay(max_prototype=10)

    def repre():
        proto.build(feats, labels, range(C_OLD))
        proto.staged()

    def step():
        repre()
        cov_pass()
        opt.step()

    def timed(fn):
        for _ in range(3):
            fn()
        hooks.join()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        hooks.join()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    res = {False: {}, True: {}}
    for _ in range(rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            for key, fn in (("ms_per_step", step), ("cov_pass_ms", cov_pass),
                            ("sgd_step_ms", opt.step), ("repre_build_ms", repre)):
                res[det].setdefault(key, []).append(timed(fn))
            if det:
                slots = sum(js.group.n_problems[3] for js in hooks._sets if js.group is not None)
                plan = opt._plans[0]["plan"]
                res[det]["slot_bytes_cov_pass"] = slots * SLOT_BYTES
                res[det]["slot_bytes_sgd_step"] = (plan.group.n_problems[3] +
                                                   plan.group2.n_problems[3]) * SLOT_BYTES
    torch.use_deterministic_algorithms(False)

    def summary(d):
        out = {}
        for k, v in d.items():
            out[k] = ({"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v)}
                      if isinstance(v, list) else v)
        return out

    print(json.dumps({"gpu": gpu_info(), "config": cfg["name"], "batch": B, "input": [H, W],
                      "rounds": rounds, "steps": steps, "off": summary(res[False]),
                      "on": summary(res[True])}))


if __name__ == "__main__":
    main()
