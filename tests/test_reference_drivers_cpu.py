"""Boundary proof: the REFERENCE'S OWN drivers -- ``demos/demo_inference.py::DemoInference`` (demo.py's tracker object) and
``siammot/engine/inferencer.py::do_inference`` (tools/test_net.py's per-video loop) -- imported UNCHANGED from /root/reference,
run once on the reference model (CPU, over the maskrcnn_benchmark stand-in) and once on the B200 engine selected by the import
switch of INTEGRATION.md section A (``SIAMMOT_ENGINE=b200`` + ``import siammot_b200.dropin``), and compared.

The engine runs over the C-ABI emulator here (there is no GPU in this container), i.e. what is proven is the BOUNDARY: that
the drivers' calls -- build_siammot(cfg), DetectronCheckpointer(cfg, model).load(path), model.to(device), model.eval(),
model(frame.to(device)), model(video_clip, given_detection=...), reset_siammot_status(), results[0].to('cpu'),
.resize(...).convert('xywh'), boxlists_to_entities(...) -- find what they expect and produce the reference's tracks
(ids exact, boxes <= 1e-3 px).  The CUDA kernels behind the same calls are pinned by the -m gpu tests.
Skipped where the reference tree does not exist (the GPU box)."""
import os
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from oracle import reference_loader  # noqa: E402

H, W, FRAMES = 192, 320, 5


def _artifacts(tmp_path):
    """What DemoInference downloads from S3 (demo_inference.py:44-72): a yaml and a checkpoint.  Here: the shipped TAO yaml with
    the test size set to the synthetic frames' size, and seeded synthetic weights in the reference's state-dict layout."""
    from siammot_b200.config import get_cfg
    from siammot_b200.synthetic import make_state_dict
    src = open(os.path.join(reference_loader.REFERENCE_ROOT, "configs", "dla", "DLA_34_FPN_EMM.yaml")).read()
    assert "MIN_SIZE_TEST: 800" in src and "MAX_SIZE_TEST: 1280" in src
    yaml_path = tmp_path / "DLA34_emm.yaml"
    yaml_path.write_text(src.replace("MIN_SIZE_TEST: 800", "MIN_SIZE_TEST: %d" % H).replace("MAX_SIZE_TEST: 1280", "MAX_SIZE_TEST: %d" % W))
    cfg = get_cfg()
    cfg.merge_from_file(str(yaml_path))
    ckpt = tmp_path / "DLA34_emm_coco_crowdhuman.pth"
    torch.save({"model": make_state_dict(cfg, 1)}, str(ckpt))
    return str(yaml_path), str(ckpt)


def _frames():
    from siammot_b200.synth_clip import make_clip_u8
    return [f.numpy() for f in make_clip_u8(FRAMES, H, W, n_obj=6, seed=0)]       # decoded RGB uint8 frames


def _neutralise_cuda(monkeypatch):
    """The drivers hard-code cuda devices (demo_inference.py:29, inferencer.py:33); there is none here."""
    orig_to = torch.Tensor.to

    def to(self, *a, **k):
        a = tuple(x for x in a if not (isinstance(x, torch.device) and x.type == "cuda") and not (isinstance(x, str) and x.startswith("cuda")))
        if isinstance(k.get("device"), (str, torch.device)) and str(k["device"]).startswith("cuda"):
            k.pop("device")
        return orig_to(self, *a, **k) if (a or k) else self
    monkeypatch.setattr(torch.Tensor, "to", to)
    monkeypatch.setattr(torch.nn.Module, "to", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)


def _import_drivers():
    reference_loader.load()
    sys.path.insert(0, os.path.join(reference_loader.REFERENCE_ROOT))
    for m in [m for m in sys.modules if m.startswith("demos") or m == "siammot.engine.inferencer"]:
        del sys.modules[m]
    from demos.demo_inference import DemoInference
    from siammot.engine.inferencer import do_inference
    return DemoInference, do_inference


def _run_demo(DemoInference, arts, frames, monkeypatch):
    monkeypatch.setattr(DemoInference, "_get_artifacts", lambda self: arts)
    from siammot.configs.defaults import cfg
    snapshot = cfg.clone()
    try:
        demo = DemoInference(gpu_id=0, track_class="person")
        out = []
        for frame_id, res in demo.process_frame_sequence(enumerate(frames)):
            out.append(dict(boxes=res.bbox.clone(), scores=res.get_field("scores").clone(), ids=res.get_field("ids").clone(),
                            labels=res.get_field("labels").clone(), mode=res.mode, size=tuple(res.size)))
        return out, type(demo.tracker).__module__
    finally:
        cfg.clear()
        cfg.update(snapshot)           # DemoInference merges into the reference's global cfg


def _run_do_inference(do_inference, arts, frames, build, monkeypatch):
    from gluoncv.torch.data.gluoncv_motion_dataset.dataset import DataSample
    from PIL import Image
    import torch.utils.data as tud
    from siammot.configs.defaults import cfg as ref_cfg
    from siammot.data.adapters.augmentation.build_augmentation import build_siam_augmentation
    cfg = ref_cfg.clone()
    cfg.merge_from_file(arts[0])
    model = build(cfg)
    from maskrcnn_benchmark.utils.checkpoint import DetectronCheckpointer
    DetectronCheckpointer(cfg, model).load(arts[1])
    # DataLoader(num_workers=4) forks workers; keep the emulation in-process
    orig = tud.DataLoader
    monkeypatch.setattr(tud, "DataLoader", lambda ds, num_workers=0, **k: orig(ds, num_workers=0, **k))
    sample = DataSample("clip0", metadata={"resolution": {"width": W, "height": H}, "fps": 30.0},
                        frames=[Image.fromarray(f, "RGB") for f in frames])
    model.reset_siammot_status()
    res = do_inference(cfg, model, sample, transforms=build_siam_augmentation(cfg, is_train=False, modality="video"))
    ents = sorted(((e.frame_num, e.id, [round(v, 3) for v in e.bbox], round(e.confidence, 4)) for e in res.entities))
    return ents, type(model).__module__


def _same_tracks(a, b):
    assert len(a) == len(b)
    for t, (x, y) in enumerate(zip(a, b)):
        assert x["mode"] == y["mode"] == "xywh" and x["size"] == y["size"] == (W, H)
        assert torch.equal(x["ids"], y["ids"]) and torch.equal(x["labels"], y["labels"]), "frame %d" % t
        if x["boxes"].numel():
            assert float((x["boxes"] - y["boxes"]).abs().max()) <= 1e-3 and float((x["scores"] - y["scores"]).abs().max()) <= 1e-3


@pytest.mark.skipif(not reference_loader.available(), reason="needs the reference's driver sources (SIAMMOT_REFERENCE_ROOT)")
def test_reference_drivers_run_unchanged_on_the_engine(monkeypatch, tmp_path):
    import cabi_emulator
    from siammot_b200 import dropin
    arts, frames = _artifacts(tmp_path), _frames()
    _neutralise_cuda(monkeypatch)
    # ---- reference model behind the reference drivers
    dropin.uninstall()
    sys.modules.pop("siammot.modelling.rcnn", None)
    DemoInference, do_inference = _import_drivers()
    ref_demo, ref_cls = _run_demo(DemoInference, arts, frames, monkeypatch)
    assert ref_cls == "siammot.modelling.rcnn"
    from siammot.modelling.rcnn import build_siammot as ref_build
    ref_ents, _ = _run_do_inference(do_inference, arts, frames, ref_build, monkeypatch)
    assert sum(int((r["ids"] >= 0).sum()) for r in ref_demo) > 0, "the scenario tracks nothing: not a test"
    # ---- the same drivers, re-imported behind the import switch: SIAMMOT_ENGINE=b200 + import siammot_b200.dropin
    cabi_emulator.install(monkeypatch)
    monkeypatch.setenv("SIAMMOT_ENGINE", "b200")
    sys.modules.pop("siammot.modelling.rcnn", None)
    assert dropin.install() is True
    try:
        DemoInference, do_inference = _import_drivers()
        eng_demo, eng_cls = _run_demo(DemoInference, arts, frames, monkeypatch)
        assert eng_cls == "siammot_b200.modelling.rcnn", "the drivers did not pick the engine up: %s" % eng_cls
        _same_tracks(ref_demo, eng_demo)
        from siammot.modelling.rcnn import build_siammot as eng_build
        eng_ents, cls2 = _run_do_inference(do_inference, arts, frames, eng_build, monkeypatch)
        assert cls2 == "siammot_b200.modelling.rcnn"
        assert [e[:2] for e in eng_ents] == [e[:2] for e in ref_ents]                       # (frame, id) of every entity
        assert np.allclose([e[2] for e in eng_ents], [e[2] for e in ref_ents], atol=2e-3) if ref_ents else True
        assert np.allclose([e[3] for e in eng_ents], [e[3] for e in ref_ents], atol=1e-3) if ref_ents else True
    finally:
        dropin.uninstall()
        for m in [m for m in sys.modules if m.startswith("demos") or m == "siammot.engine.inferencer"]:
            del sys.modules[m]


def test_dropin_switch_is_inert_without_the_environment_variable(monkeypatch):
    from siammot_b200 import dropin
    monkeypatch.delenv("SIAMMOT_ENGINE", raising=False)
    dropin.uninstall()
    assert dropin.install() is False and not getattr(sys.modules.get("siammot.modelling.rcnn"), "__siammot_b200__", False)
