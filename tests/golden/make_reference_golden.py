"""Store what the module-level comparisons with the reference compare against: tests/golden/reference_modules.pt.gz.

Runs the UNMODIFIED reference (siammot/modelling/**, siammot/utils/boxlists_to_entities.py, siammot/engine/inferencer.py) on
the CPU over the maskrcnn_benchmark stand-in in oracle/shim, like make_golden.py; the reference tree is located by
oracle/reference_loader.py (SIAMMOT_REFERENCE_ROOT):

    python tests/golden/make_reference_golden.py

Stored (inputs and weights are not: they are pure functions of the seeds the tests use):
  * xcorr       -- the reference's depthwise correlation on seeded inputs, a fixed sample of its output;
  * dla         -- per DLA body (and deformable variant): the reference module's state-dict keys and shapes, and a fixed
                   sample of each of its four output maps on seeded weights and input (64x96);
  * layout      -- the state-dict keys and shapes of the reference's whole SiamMOT for four scenarios and detector-only;
  * egress      -- the entities the reference's per-frame result path makes of seeded results, for three video sizes;
  * postprocess -- the (id, frame, box) keys DatasetInference._postprocess_tracks keeps of a seeded clip.
"""
import ast
import gzip
import io
import os
import sys
import textwrap

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

from oracle import reference_loader  # noqa: E402

OUT = os.path.join(HERE, "reference_modules.pt.gz")     # the key lists compress ~5x
SAMPLE = 256                  # stored elements per output map


def sample(t, n=SAMPLE, seed=0):
    """A fixed, seeded sample of a tensor's elements: flat indices and their values."""
    flat = t.detach().reshape(-1)
    idx = torch.randint(0, flat.numel(), (min(n, flat.numel()),), generator=torch.Generator().manual_seed(seed))
    return dict(shape=tuple(t.shape), idx=idx.int(), val=flat[idx].clone())


def xcorr():
    from siammot.modelling.track_head.EMM.xcorr import xcorr_depthwise
    from test_oracle_golden import xcorr_inputs
    return sample(xcorr_depthwise(*xcorr_inputs()), 2048)


def dla():
    from siammot.modelling.backbone import dla as ref_dla
    from test_oracle_dla_family_cpu import CASES, seeded_weights
    out = {}
    for arch, dcn in CASES:
        torch.manual_seed(0)
        net = ref_dla.BACKBONE[arch](dcn).eval()
        sd = net.state_dict()
        keys = [(k, tuple(v.shape)) for k, v in sd.items()]
        weights, x = seeded_weights(keys)
        net.load_state_dict(weights, strict=True)
        with torch.no_grad():
            maps = net(x)
        out[(arch, dcn)] = dict(keys=keys, maps=[sample(m, seed=i) for i, m in enumerate(maps)])
        print(arch, dcn, [tuple(m.shape) for m in maps])
    return out


def layout():
    from scenarios import ORACLE_SCENARIOS, SCENARIOS
    from test_host_cpu import LAYOUT_SCENARIOS
    cfg0, build = reference_loader.load()

    def keys(yaml, overrides):
        rcfg = cfg0.clone()
        rcfg.merge_from_file(os.path.join(reference_loader.REFERENCE_ROOT, "configs", "dla", yaml))
        rcfg.merge_from_list(overrides)
        rcfg.MODEL.DEVICE = "cpu"
        return [(k, tuple(v.shape)) for k, v in build(rcfg).state_dict().items()]
    out = {}
    for name in LAYOUT_SCENARIOS:
        sc = SCENARIOS.get(name) or ORACLE_SCENARIOS[name]
        out[name] = keys(sc["yaml"], sc["overrides"])
    out["detector_only"] = keys("DLA_34_FPN_EMM.yaml", ["MODEL.TRACK_ON", False])
    return out


def _entity(e):
    return dict(bbox=[float(v) for v in e.bbox], confidence=float(e.confidence), labels=e.labels, id=int(e.id),
                frame_num=int(e.frame_num), time=float(e.time))


def egress():
    from maskrcnn_benchmark.structures.bounding_box import BoxList as RefBoxList
    from siammot.utils.boxlists_to_entities import boxlists_to_entities
    from test_egress_cpu import CLASSES, VIDEOS, random_results
    out = {}
    for video in VIDEOS:
        ents = []
        for t, r in enumerate(random_results(video[0])):          # the reference path, per frame (inferencer.py:64-70)
            rb = RefBoxList(r.bbox.clone(), r.size, "xyxy")
            for f in r.fields():
                rb.add_field(f, r.get_field(f))
            o = rb.resize([video[0], video[1]]).convert("xywh").to(torch.device("cpu"))
            ents += boxlists_to_entities([o], 100 + t, [0.04 * (100 + t)], class_table=list(CLASSES))
        out[video] = [_entity(e) for e in ents]
    return out


def postprocess():
    """DatasetInference._postprocess_tracks, literally, from the reference file (its module needs motmetrics & co. to import)."""
    from gluoncv.torch.data.gluoncv_motion_dataset.dataset import DataSample
    from siammot_b200 import egress as eg
    from test_egress_cpu import CLASSES, POSTPROCESS, random_results
    src = open(os.path.join(reference_loader.REFERENCE_ROOT, "siammot", "engine", "inferencer.py")).read()
    node = next(n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == "_postprocess_tracks")
    ns = {"np": np, "DataSample": DataSample}
    exec(textwrap.dedent(ast.get_source_segment(src, node)), ns)

    class Self(object):
        _track_len, _track_conf = POSTPROCESS["track_len"], POSTPROCESS["track_conf"]
    tracks = eg.clip_to_tracks(random_results(POSTPROCESS["seed"], n_frames=POSTPROCESS["frames"]), 1280, 720)
    kept = ns["_postprocess_tracks"](Self(), DataSample("v", entities=eg.to_entities(tracks, list(CLASSES)))).entities
    return sorted((int(e.id), int(e.frame_num), tuple(float(v) for v in e.bbox)) for e in kept)


if __name__ == "__main__":
    reference_loader.load()
    gold = dict(torch=torch.__version__, xcorr=xcorr(), dla=dla(), layout=layout(), egress=egress(), postprocess=postprocess())
    buf = io.BytesIO()
    torch.save(gold, buf)
    with gzip.open(OUT, "wb") as f:
        f.write(buf.getvalue())
    print("wrote", OUT, os.path.getsize(OUT), "bytes")
