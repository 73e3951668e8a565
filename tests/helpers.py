import gzip
import io
import os

import torch

from scenarios import ORACLE_SCENARIOS, SCENARIOS, golden_path, inject_boxes
from siammot_b200.config import get_cfg
from siammot_b200.synthetic import make_state_dict
from siammot_b200.synth_clip import make_clip

CONFIG_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "siammot_b200", "configs")
YAML_MAP = {"DLA_34_FPN_EMM.yaml": "dla34_emm.yaml", "DLA_34_FPN_EMM_MOT17.yaml": "dla34_emm_mot17.yaml",
            "DLA_34_FPN_EMM_AOT.yaml": "dla34_emm_aot.yaml"}


def _spec(name):
    return SCENARIOS.get(name) or ORACLE_SCENARIOS[name]


def scenario_cfg(name):
    sc = _spec(name)
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(CONFIG_DIR, YAML_MAP[sc["yaml"]]))
    cfg.merge_from_list(sc["overrides"])
    return cfg


def scenario_inputs(name):
    sc = _spec(name)
    cfg = scenario_cfg(name)
    return cfg, make_state_dict(cfg, sc["weight_seed"]), make_clip(sc["frames"], sc["H"], sc["W"], sc["n_obj"], sc["clip_seed"])


def load_golden(name):
    """tests/golden/<name>.pt, or <name>.pt.gz where the fixture compresses well."""
    path = golden_path(name)
    if not os.path.exists(path):
        with gzip.open(path + ".gz", "rb") as f:
            return torch.load(io.BytesIO(f.read()), weights_only=False)
    return torch.load(path, weights_only=False)


def run_oracle_scenario(name):
    """Run the CPU oracle over a scenario; returns list of per-frame dicts (+ trace)."""
    from oracle.siammot_oracle import OracleSiamMOT, build_memory
    sc = _spec(name)
    cfg, sd, clip = scenario_inputs(name)
    orc = OracleSiamMOT(cfg, sd)
    orc.reset()
    start = 0
    if sc["inject"] is not None:
        feats = orc.features(clip[0])
        boxes = inject_boxes(sc["inject"])
        ids = torch.tensor([orc.pool.start() for _ in range(len(boxes))])
        det = dict(boxes=boxes, scores=torch.full((len(boxes),), 0.9), ids=ids,
                   labels=torch.ones(len(boxes), dtype=torch.int64))
        orc.memory = build_memory(orc.P, cfg, orc.pool, feats, det)
        orc.pool.frame += 1
        start = 1
    out = []
    for t in range(start, sc["frames"]):
        det = orc.forward(clip[t])
        rec = dict(det)
        rec["trace"] = orc.trace
        rec["active"] = sorted(orc.pool.active)
        rec["dormant"] = sorted(orc.pool.dormant.keys())
        out.append(rec)
    return out
