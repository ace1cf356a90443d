"""The mmengine / mmdet branch of ``registry.register_all`` executed against fabricated
``mmengine.registry`` / ``mmdet.*`` modules (neither package is installable here): the
drop-ins must land in OPTIMIZERS / MODELS / RUNNERS under the reference's names, bound onto
the reference's own base classes, and build from the reference's config dicts.  Runs in a
subprocess so that the fabricated modules never leak into other tests."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = textwrap.dedent('''
    import sys, types, json
    import torch

    class Registry:                                   # the part of mmengine.Registry used here
        def __init__(self, name):
            self.name, self.module_dict = name, {}
        def register_module(self, name=None, module=None, force=False):
            if name in self.module_dict and not force:
                raise KeyError("%s is already registered in %s" % (name, self.name))
            self.module_dict[name] = module
            return module
        def build(self, cfg, **kw):
            cfg = dict(cfg)
            return self.module_dict[cfg.pop("type")](**cfg, **kw)

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        m.__path__ = []
        sys.modules[name] = m
        return m

    OPTIMIZERS, MODELS, RUNNERS = Registry("optimizer"), Registry("model"), Registry("runner")

    class RefOptim: pass
    class RefRoIHead(torch.nn.Module):                # stands for mmdet's StandardRoIHead
        def __init__(self, bbox_head=None, **kw):
            super().__init__()
            self.bbox_head = bbox_head
            self.with_shared_head = False
        def loss(self, x, rpn_results_list, batch_data_samples):
            return {"loss_cls": torch.tensor(1.0)}
    class RefSampledHead(RefRoIHead):                 # the fork's StandardRoIReplayHead (:31-69)
        def __init__(self, *a, previous_path=None, **kw):
            super().__init__(*a, **kw)
            self.replay, self.counter, self.ref_previous_path = False, [0] * 80, previous_path
        def loss(self, x, rpn_results_list, batch_data_samples, replay=True):
            assert replay is False, "the fork's CPU replay branch must not run"
            return super().loss(x, rpn_results_list, batch_data_samples)
        def get_bbox_stuff(self, *a, **k):
            return "fork"
    class RefRunner:                                  # the fork's BRNullSpaceRunner
        def cal_rois(self): return "fork"
        def cal_fea_in(self, loader): raise AssertionError("reference cal_fea_in called")

    OPTIMIZERS.register_module(name="SGDNSCL", module=RefOptim)
    MODELS.register_module(name="StandardRoIReplayHead", module=RefSampledHead)
    MODELS.register_module(name="StandardMultiPrototypeReplayHead", module=RefSampledHead)
    RUNNERS.register_module(name="BRNullSpaceRunner", module=RefRunner)
    mod("mmengine"); mod("mmengine.registry", OPTIMIZERS=OPTIMIZERS)
    mod("mmengine.model", is_model_wrapper=lambda m: False)
    mod("mmdet"); mod("mmdet.registry", MODELS=MODELS, RUNNERS=RUNNERS)
    mod("mmdet.models"); mod("mmdet.models.roi_heads")
    mod("mmdet.models.roi_heads.standard_roi_replay_head", StandardRoIReplayHead=RefSampledHead)
    mod("mmdet.engine"); mod("mmdet.engine.runner")
    mod("mmdet.engine.runner.nsrunner_roi_replay", BRNullSpaceRunner=RefRunner)

    import nsgp_repre_b200 as pkg
    # importing the package touches the local table only
    assert OPTIMIZERS.module_dict["SGDNSCL"] is RefOptim and not pkg.registry.MM_REGISTERED
    try:
        pkg.registry.register_all(force=False, strict=True)
        raise SystemExit("force=False must not replace an existing entry silently")
    except KeyError:
        pass
    import nsgp_repre_b200.mm                         # the custom_imports hook: force + strict
    reg = pkg.registry.MM_REGISTERED
    assert reg == {"OPTIMIZERS": ["SGDNSCL"],
                   "MODELS": ["StandardRoIReplayHead", "StandardMultiPrototypeReplayHead"],
                   "RUNNERS": ["BRNullSpaceRunner"]}, reg
    assert pkg.registry.MMENGINE_AVAILABLE

    cfg = json.load(open(sys.argv[1]))
    opt = OPTIMIZERS.build(cfg["optim_wrapper"]["optimizer"],
                           params=[torch.nn.Parameter(torch.zeros(2, 2))])
    assert isinstance(opt, pkg.SGDNSCL) and opt.defaults["svd"] is True

    Runner = RUNNERS.module_dict[cfg["runner_type"]]
    assert issubclass(Runner, RefRunner) and issubclass(Runner, pkg.NullSpaceRunnerMixin)
    assert Runner.cal_fea_in is pkg.NullSpaceRunnerMixin.cal_fea_in
    assert Runner.compute_cov is pkg.NullSpaceRunnerMixin.compute_cov
    assert Runner().cal_rois() == "fork"              # everything else stays the fork's

    head_cfg = dict(cfg["tasks"]["cl_faster_rcnn_nsgp_repre_19_1_2.py"]["roi_head"])
    head_cfg["previous_path"] = "/nonexistent/x_1"    # no artifacts: replay stays off
    head = MODELS.build(head_cfg, bbox_head=torch.nn.Identity())
    assert isinstance(head, RefSampledHead) and isinstance(head, pkg.prototypes.ReplayHeadMixin)
    assert head.replay is False and head.task_split == [0, 19, 20] and head.max_proto == 10
    assert head.ref_previous_path is None             # the fork never loads onto the CPU
    assert head.get_bbox_stuff() == "fork" and head.counter == [0] * 80
    assert set(head.loss(None, None, None)) == {"loss_cls"}
    sampled = MODELS.build(dict(type="StandardRoIReplayHead", previous_path=None),
                           bbox_head=torch.nn.Identity())
    assert sampled.replay is False and set(sampled.loss(None, None, None)) == {"loss_cls"}
    assert type(sampled).replay_loss is pkg.prototypes.ReplayHeadMixin.teacher_replay_loss
    print("fake-mm registration ok")
''')


def test_register_all_into_fabricated_mm_registries(tmp_path):
    script = tmp_path / "fake_mm.py"
    script.write_text(SCRIPT)
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, str(script),
                          os.path.join(ROOT, "tests", "golden", "ref_cfg_keys.json")],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "fake-mm registration ok" in out.stdout
