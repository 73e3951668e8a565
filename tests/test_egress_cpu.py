"""Clip-level result egress (siammot_b200/egress.py) against the reference's own code: what ``boxlists_to_entities`` (behind the
per-frame resize / convert of inferencer.py:64-70) and ``DatasetInference._postprocess_tracks`` make of seeded results is stored
in tests/golden/reference_modules.pt.gz (tests/golden/make_reference_golden.py runs both on the reference)."""
import pytest
import torch

from helpers import load_golden

CLASSES = ("person", "vehicle")
VIDEOS = [(1280, 720), (1920, 1080), (2560, 1408)]
POSTPROCESS = dict(seed=7, frames=40, track_len=5, track_conf=0.7)


def random_results(seed, n_frames=12, net=(1280, 704)):
    from siammot_b200.structures import BoxList
    g = torch.Generator().manual_seed(seed)
    out = []
    for t in range(n_frames):
        n = int(torch.randint(0, 9, (1,), generator=g))
        xy = torch.rand(n, 2, generator=g) * torch.tensor([net[0] * 0.8, net[1] * 0.8])
        wh = torch.rand(n, 2, generator=g) * 200 + 5
        bl = BoxList(torch.cat([xy, xy + wh], 1), net, "xyxy")
        bl.add_field("scores", torch.rand(n, generator=g) * 0.5 + 0.5)
        bl.add_field("ids", torch.randint(-1, 4, (n,), generator=g))
        bl.add_field("labels", torch.randint(1, 3, (n,), generator=g))
        out.append(bl)
    return out


@pytest.mark.parametrize("video", VIDEOS)
def test_clip_to_tracks_and_entities_equal_the_reference_path(video):
    from siammot_b200 import egress
    ref_entities = load_golden("reference_modules")["egress"][video]
    results = random_results(video[0])
    tracks = egress.clip_to_tracks(results, video[0], video[1], first_frame_idx=100, timestamps=[0.04 * (100 + t) for t in range(len(results))])
    got = egress.to_entities(tracks, class_table=list(CLASSES))
    assert len(got) == len(ref_entities) == len(tracks)
    for a, b in zip(got, ref_entities):
        assert a.bbox == b["bbox"] and a.confidence == b["confidence"] and a.labels == b["labels"]
        assert a.id == b["id"] and a.frame_num == b["frame_num"] and a.time == b["time"]


def test_postprocess_tracks_equals_the_reference_filter():
    from siammot_b200 import egress
    ref = load_golden("reference_modules")["postprocess"]
    tracks = egress.clip_to_tracks(random_results(POSTPROCESS["seed"], n_frames=POSTPROCESS["frames"]), 1280, 720)
    got = egress.to_entities(egress.postprocess_tracks(tracks, POSTPROCESS["track_len"], POSTPROCESS["track_conf"]), list(CLASSES))
    key = lambda e: (e.id, e.frame_num, tuple(e.bbox))
    assert len(ref) > 0 and ref == sorted(map(key, got))
    assert all(e.id >= 0 for e in got)
    # grouped by id, frames ascending
    assert [(e.id, e.frame_num) for e in got] == sorted((e.id, e.frame_num) for e in got)
