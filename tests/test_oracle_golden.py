"""Pin the CPU oracle (oracle/siammot_oracle.py) against the reference.

The golden vectors were produced by the reference's own modules (tests/golden/make_golden.py).
Tolerance: both sides are fp32 CPU PyTorch built from the same primitive ops, so they agree to
rounding; 1e-4 px / 1e-5 score leaves room for a different CPU / oneDNN code path."""
import pytest
import torch

from helpers import load_golden, run_oracle_scenario
from scenarios import ORACLE_SCENARIOS, SCENARIOS

def _canon(boxes, obj):
    rows = sorted(range(boxes.shape[0]), key=lambda i: (-float(obj[i]),) + tuple(boxes[i].tolist()))
    return boxes[rows]


BOX_TOL = 1e-4
SCORE_TOL = 1e-5


@pytest.mark.parametrize("name", list(SCENARIOS) + list(ORACLE_SCENARIOS))
def test_oracle_matches_reference_golden(name):
    gold = load_golden(name)["frames"]
    got = run_oracle_scenario(name)
    assert len(got) == len(gold)
    for t, (g, o) in enumerate(zip(gold, got)):
        assert o["boxes"].shape == g["boxes"].shape, "frame %d: box count" % t
        assert torch.equal(o["ids"], g["ids"]), "frame %d: ids must be bit-exact" % t
        assert torch.equal(o["labels"], g["labels"])
        assert (o["boxes"] - g["boxes"]).abs().max() <= BOX_TOL
        assert (o["scores"] - g["scores"]).abs().max() <= SCORE_TOL
        assert o["active"] == g["active"] and o["dormant"] == g["dormant"]
        # proposals: the order inside a group of EQUAL fp32 objectness is implementation-defined in
        # the reference (torch.topk); compare after a canonical sort inside such groups
        props = _canon(o["trace"]["proposals"][:32], g["objectness"])
        assert (props - _canon(g["props"], g["objectness"])).abs().max() <= BOX_TOL
        if "track_boxes" in g:
            tr = o["trace"]["tracks"]
            assert torch.equal(tr["ids"], g["track_ids"])
            assert (tr["boxes"] - g["track_boxes"]).abs().max() <= BOX_TOL
            assert (tr["scores"] - g["track_scores"]).abs().max() <= SCORE_TOL


def test_golden_scenarios_exercise_the_state_machine():
    """The fixtures are only useful if tracks start, persist, go dormant, resume and expire."""
    g = load_golden("emm_256x384")["frames"]
    ids_per_frame = [set(f["ids"][f["ids"] >= 0].tolist()) for f in g]
    assert all(len(s) > 0 for s in ids_per_frame)
    assert any(ids_per_frame[t] & ids_per_frame[t + 1] for t in range(len(g) - 1)), "no track persisted"
    assert any(len(f["dormant"]) > 0 for f in g)
    resumed = any((set(g[t]["dormant"]) & set(g[t + 1]["active"])) for t in range(len(g) - 1))
    assert resumed, "no dormant track was resumed"
    e = load_golden("emm_amodal_expire_192x320")["frames"]
    seen, expired = set(), False
    for f in e:
        alive = set(f["active"]) | set(f["dormant"])
        expired |= bool(seen - alive)
        seen |= alive
    assert expired, "no track expired"


def xcorr_inputs():
    torch.manual_seed(0)
    return torch.randn(5, 16, 30, 30), torch.randn(5, 16, 15, 15)


def test_oracle_matches_reference_xcorr():
    """The restatement of xcorr.py (pure torch) against the reference's own output on the same inputs
    (tests/golden/make_reference_golden.py stores a fixed sample of it)."""
    from oracle.siammot_oracle import xcorr_depthwise
    gold = load_golden("reference_modules")["xcorr"]
    got = xcorr_depthwise(*xcorr_inputs())
    assert tuple(got.shape) == gold["shape"]
    assert torch.equal(got.reshape(-1)[gold["idx"].long()], gold["val"])


def test_oracle_matches_reference_golden_with_given_detections():
    """Public-detection path (roi_heads.py:26-34): the reference was fed `given_detection` every frame, one frame with an
    empty list (tests/golden/make_golden.py run_given)."""
    from helpers import CONFIG_DIR, YAML_MAP
    from oracle.siammot_oracle import OracleSiamMOT
    from scenarios import GIVEN_SCENARIOS, given_boxes
    from siammot_b200.config import get_cfg
    from siammot_b200.synth_clip import make_clip
    from siammot_b200.synthetic import make_state_dict
    import os
    name = "given_det_192x320"
    sc = GIVEN_SCENARIOS[name]
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(CONFIG_DIR, YAML_MAP[sc["yaml"]]))
    cfg.merge_from_list(sc["overrides"])
    gold = load_golden(name)["frames"]
    orc = OracleSiamMOT(cfg, make_state_dict(cfg, sc["weight_seed"]))
    orc.reset()
    clip = make_clip(sc["frames"], sc["H"], sc["W"], sc["n_obj"], sc["clip_seed"])
    tracked = 0
    for t, (boxes, g) in enumerate(zip(given_boxes(sc), gold)):
        n = boxes.shape[0]
        given = dict(boxes=boxes, scores=torch.ones(n), ids=torch.full((n,), -1, dtype=torch.int64),
                     labels=torch.ones(n, dtype=torch.int64))
        o = orc.forward(clip[t], given_detection=given)
        assert o["boxes"].shape == g["boxes"].shape, "frame %d: box count" % t
        assert torch.equal(o["ids"], g["ids"]), "frame %d: ids must be bit-exact" % t
        assert torch.equal(o["labels"], g["labels"])
        if o["boxes"].numel():
            assert (o["boxes"] - g["boxes"]).abs().max() <= BOX_TOL
            assert (o["scores"] - g["scores"]).abs().max() <= SCORE_TOL
        assert sorted(orc.pool.active) == g["active"] and sorted(orc.pool.dormant.keys()) == g["dormant"]
        tracked += int((g["ids"] >= 0).sum())
    assert tracked >= 10


def test_full_size_fixture_is_decisive_and_the_oracle_reproduces_it():
    """tests/golden/full_720p30.pt (the reference on the benchmark geometry: 3x704x1280, 30 injected tracks, tweaked head weights):
    the stored decision margins clear the floors the GPU test demands, and the CPU oracle reproduces the reference's first frames
    (the generator checked all of them when it wrote the fixture)."""
    import fp16_scene as fs
    from decisive import MarginOracle
    from scenarios import FULL_SCENARIOS
    from test_fp16_e2e_gpu import MARGIN_FLOOR
    name = "full_720p30"
    sc = FULL_SCENARIOS[name]
    gold = load_golden(name)
    assert len(gold["frames"]) == sc["frames"] - 1 >= 8 and len(gold["margins"]) == len(gold["frames"])
    for t, m in enumerate(gold["margins"]):
        for k, floor in MARGIN_FLOOR.items():
            assert m[k] >= floor, (t, k, m[k])
    assert all(int((f["ids"] >= 0).sum()) >= sc["tracks"] for f in gold["frames"])       # the injected tracks live on, one is born
    scene = fs.build_scene(sc["weight_seed"], sc["clip_seed"], 2, sc["tweak"], workload=sc["workload"], tracks=sc["tracks"], n_obj=sc["n_obj"])
    mo = MarginOracle(scene["cfg"], scene["sd"])
    mo.inject(scene["clip"][0], scene["boxes"])
    for t in (1, 2):
        out, m = mo.step(scene["clip"][t])
        ref = gold["frames"][t - 1]
        assert torch.equal(out["ids"], ref["ids"]) and torch.equal(out["labels"], ref["labels"])
        assert float((out["boxes"] - ref["boxes"]).abs().max()) <= 1e-3
        assert abs(m["det_thresh"] - gold["margins"][t - 1]["det_thresh"]) <= 1e-4
