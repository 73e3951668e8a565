"""CPU-only checks of the host side: C-ABI library loads and exports every symbol smot.h declares,
config surface, BoxList semantics, track pool state machine (no compute calls without a GPU)."""
import ctypes
import os
import re

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    path = __graft_entry__.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(REPO, "include", "smot.h")).read()
    names = set(re.findall(r"\b(smot_[a-z0-9_]+)\s*\(", header))
    assert len(names) >= 15
    for n in sorted(names):
        assert hasattr(lib, n), "libsmot.so does not export %s" % n
    from siammot_b200 import _lib
    assert _lib.lib().smot_abi_version() == _lib.ABI_VERSION


def test_argument_errors_are_reported_not_crashed():
    from siammot_b200 import _lib
    l = _lib.lib()
    d = _lib.ConvDesc()
    assert l.smot_conv2d(ctypes.byref(d), None) == 1  # SMOT_ERR_INVALID: null tensors
    assert b"null" in l.smot_last_error()
    assert l.smot_sort_nms(None, 4, None, 1, None, 5000, 0.0, 0.5, 10, 0, None, None, None, None, None, None, 0, None) == 1


def test_product_does_not_import_the_oracle():
    for root, _, files in os.walk(os.path.join(REPO, "siammot_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_no_undefined_names_in_host_code():
    """The GPU-side host paths cannot run in a container without a GPU; at least no name in them is unbound."""
    import sys
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import lint_names
    bad = [(os.path.relpath(f, REPO), line, name) for f in lint_names.default_files() for line, name in lint_names.undefined_names(f)]
    assert not bad, bad


def test_bench_workloads_resolve_to_the_stated_network_sizes():
    """bench.py's --workload table: the cfg overrides give exactly the network input size the workload text states."""
    import sys
    sys.path.insert(0, REPO)
    import bench
    from siammot_b200.preprocess import get_size
    try:
        for name, w in bench.WORKLOADS.items():
            bench.select_workload(name)
            cfg = bench.build_cfg("float16")
            h, wd = w["src"]
            assert get_size(wd, h, cfg.INPUT.MIN_SIZE_TEST, cfg.INPUT.MAX_SIZE_TEST, cfg.DATALOADER.SIZE_DIVISIBILITY) == w["net"]
            assert bench.track_table().shape == (w["tracks"], 4)
            assert "%dx%d" % w["net"] in w["text"] and str(w["tracks"]) in w["text"]
        # the default workload's track table is the one every committed bench line was measured on
        bench.select_workload("720p30")
        t = bench.track_table()
        assert t.shape == (30, 4) and abs(float(t.sum()) - 58072.671875) < 0.01
    finally:
        bench.select_workload("720p30")


def test_config_loads_reference_style_yaml_and_overrides():
    from siammot_b200.config import get_cfg
    cfg = get_cfg()
    assert cfg.MODEL.TRACK_HEAD.MAX_DORMANT_FRAMES == 1 and cfg.MODEL.RPN.POST_NMS_TOP_N_TEST == 300
    cfg.merge_from_file(os.path.join(REPO, "siammot_b200", "configs", "dla34_emm_mot17.yaml"))
    assert cfg.INPUT.AMODAL is True and cfg.MODEL.TRACK_HEAD.MAX_DORMANT_FRAMES == 30
    cfg.merge_from_list(["MODEL.TRACK_HEAD.TRACK_THRESH", 0.5, "SOLVER.STEPS", "(1, 2)"])
    assert cfg.MODEL.TRACK_HEAD.TRACK_THRESH == 0.5 and cfg.SOLVER.STEPS == (1, 2)
    c2 = cfg.clone()
    c2.MODEL.TRACK_HEAD.TRACK_THRESH = 0.1
    assert cfg.MODEL.TRACK_HEAD.TRACK_THRESH == 0.5
    cfg.freeze()
    with pytest.raises(AttributeError):
        cfg.DTYPE = "float16"


def test_boxlist_legacy_semantics():
    from siammot_b200.structures import BoxList, cat_boxlist, remove_small_boxes
    b = BoxList(torch.tensor([[10., 20., 29., 59.], [-5., -5., 700., 800.], [3., 3., 3., 3.]]), (640, 480))
    assert b.area().tolist() == [20 * 40, 706 * 806, 1]
    x = b.convert("xywh")
    assert x.bbox[0].tolist() == [10., 20., 20., 40.] and torch.equal(x.convert("xyxy").bbox, b.bbox)
    c = BoxList(b.bbox.clone(), (640, 480)).clip_to_image(remove_empty=True)
    assert c.bbox.tolist() == [[10., 20., 29., 59.], [0., 0., 639., 479.]]
    b.add_field("scores", torch.tensor([0.1, 0.2, 0.3]))
    r = b.resize((1280, 960))
    assert r.bbox[0].tolist() == [20., 40., 58., 118.] and r.size == (1280, 960)
    assert len(cat_boxlist([b, b])) == 6 and len(remove_small_boxes(b, 2)) == 2
    assert len(b[torch.tensor([True, False, True])]) == 2


def test_track_pool_state_machine():
    from siammot_b200.modelling.track_utils import TrackPool, TrackUtils
    p = TrackPool(max_dormant_frames=2)
    a, b, c = p.start_track(), p.start_track(), p.start_track()
    assert (a, b, c) == (0, 1, 2) and p.get_active_ids() == {0, 1, 2}
    p.increment_frame()
    p.suspend_track(1)
    assert p.get_dormant_ids() == {1} and p._dormant_ids[1] == 0
    with pytest.raises(ValueError):
        p.suspend_track(1)
    p.expire_tracks()          # frame 1 - last 0 = 1 < 2: stays
    assert p.get_dormant_ids() == {1}
    p.increment_frame()
    p.expire_tracks()          # 2 - 0 >= 2: expires
    assert p.get_dormant_ids() == set()
    with pytest.raises(ValueError):
        p.resume_track(1)
    p.suspend_track(2)
    p.resume_track(2)
    assert p.get_active_ids() == {0, 2} and p.start_track() == 3
    p.reset()
    assert p.start_track() == 0
    tu = TrackUtils(search_expansion=1.0, min_search_wh=0, pad_pixels=512)
    sr = tu.search_region(torch.tensor([[100., 100., 159., 249.]]))
    assert sr.tolist() == [[582., 537., 701., 836.]]


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_host_solver_matches_oracle_on_random_sequences(seed):
    """The product's host half of the solver (numpy, NMS survivors in, ids out) and its TrackPool against the oracle's
    TrackSolver.forward restatement over 40 random frames: ids, folded scores and the pool state (active set, dormant
    table incl. insertion order, id counter) must agree exactly every frame."""
    import numpy as np
    from oracle import prims
    from oracle.siammot_oracle import PoolState, solver_forward
    from siammot_b200.config import get_cfg
    from siammot_b200.modelling.rcnn import TrackSolver
    from siammot_b200.modelling.track_utils import TrackPool
    cfg = get_cfg()
    T = cfg.MODEL.TRACK_HEAD
    T.MAX_DORMANT_FRAMES = 3
    g = torch.Generator().manual_seed(seed)
    pool_o = PoolState(T.MAX_DORMANT_FRAMES)
    pool_p = TrackPool(max_dormant_frames=T.MAX_DORMANT_FRAMES)
    solver = TrackSolver(pool_p, T.TRACK_THRESH, T.START_TRACK_THRESH, T.RESUME_TRACK_THRESH)
    started = 0
    for t in range(40):
        # candidates: fresh detections (id -1, score in (0.05, 1)) + one row per track in memory (active and dormant,
        # score = refined average in [1, 2)); boxes cluster so that NMS removes some rows, tracks included
        known = sorted(pool_o.active) + list(pool_o.dormant.keys())
        n_det = int(torch.randint(3, 12, (1,), generator=g))
        ctr = torch.rand(n_det + len(known), 2, generator=g) * 60 + torch.randint(0, 3, (n_det + len(known), 1), generator=g) * 200
        wh = torch.rand(n_det + len(known), 2, generator=g) * 20 + 50
        boxes = torch.cat([ctr, ctr + wh], 1)
        scores = torch.cat([torch.rand(n_det, generator=g) * 0.95 + 0.05, 1.0 + torch.rand(len(known), generator=g)])
        if len(known):   # exact ties between a detection and a track row, and scores straddling the thresholds
            scores[n_det] = 1.0 + scores[0]
        ids = torch.tensor([-1] * n_det + known, dtype=torch.int64)
        labels = torch.ones(n_det + len(known), dtype=torch.int64)
        det = dict(boxes=boxes, scores=scores.clone(), ids=ids.clone(), labels=labels)
        ref = solver_forward(cfg, pool_o, det)
        # the product path: active +1 and NMS happen on the device (track_combine / sort_nms kernels); emulate them with the
        # same primitives, then the host half under test
        active = pool_p.get_active_ids()
        adj = scores + torch.tensor([1.0 if int(i) in active else 0.0 for i in ids])
        keep = prims.nms_legacy(boxes, adj, 0.5)
        all_track_ids = set(ids[ids >= 0].tolist())
        sc, out_ids = solver.resolve(adj[keep].numpy(), ids[keep].numpy(), all_track_ids)
        assert out_ids.tolist() == ref["ids"].tolist(), "frame %d" % t
        assert np.array_equal(sc, ref["scores"].numpy()), "frame %d" % t
        assert pool_p.get_active_ids() == pool_o.active and list(pool_p._dormant_ids.items()) == list(pool_o.dormant.items())
        assert pool_p._max_id + 1 == pool_o.next_id and pool_p._frame_idx == pool_o.frame
        started = pool_o.next_id
    assert started > 10 and len(pool_o.dormant) + len(pool_o.active) > 0


def test_search_region_numpy_twin_is_bit_exact():
    """TrackUtils.search_region_np (the per-frame host path) against the torch method and the oracle restatement."""
    import numpy as np
    from oracle.siammot_oracle import search_region
    from siammot_b200.modelling.track_utils import TrackUtils
    g = torch.Generator().manual_seed(4)
    for exp, min_wh in ((1.0, 0), (1.0, 120), (4.0, 0)):
        tu = TrackUtils(search_expansion=exp, min_search_wh=min_wh, pad_pixels=512)
        xy = torch.rand(200, 2, generator=g) * 1200 - 100
        wh = torch.rand(200, 2, generator=g) * 400 + 1
        boxes = torch.cat([xy, xy + wh], 1)
        ref = search_region(boxes, 512, exp, min_wh)
        assert torch.equal(tu.search_region(boxes), ref)
        assert np.array_equal(tu.search_region_np(boxes.numpy()), ref.numpy())


LAYOUT_SCENARIOS = ["emm_256x384", "emm_r50_192x320", "emm_dla102_192x320", "emm_dla60_dcn_192x320"]


def _reference_layout(name):
    """The keys and shapes of the reference's SiamMOT state dict (tests/golden/make_reference_golden.py)."""
    import sys
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import load_golden
    return dict(load_golden("reference_modules")["layout"][name])


@pytest.mark.parametrize("name", LAYOUT_SCENARIOS)
def test_state_dict_layout_equals_the_reference_module_tree(name):
    """build_siammot(cfg).state_dict() has exactly the keys and shapes of the reference's SiamMOT (DLA-34-FPN and the upstream
    R-50-FPN body), so DetectronCheckpointer-style checkpoints load unchanged."""
    from helpers import scenario_cfg
    from siammot_b200.modelling import build_siammot
    ref = _reference_layout(name)
    ours = {k: tuple(v.shape) for k, v in build_siammot(scenario_cfg(name)).state_dict().items()}
    assert ours == ref


def test_detector_only_state_dict_layout_equals_the_reference():
    """MODEL.TRACK_ON False: no roi_heads.track.* parameters on either side (roi_heads.py:87-100)."""
    ref = _reference_layout("detector_only")
    from helpers import scenario_cfg
    from siammot_b200.modelling import build_siammot
    cfg = scenario_cfg("emm_256x384")
    cfg.merge_from_list(["MODEL.TRACK_ON", False])
    ours = {k: tuple(v.shape) for k, v in build_siammot(cfg).state_dict().items()}
    assert ours == ref and not any(k.startswith("roi_heads.track") for k in ours)
