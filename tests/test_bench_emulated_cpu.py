"""bench.py's GPU arm cannot run in a container without a GPU; its control flow can: over tests/cabi_emulator.py the whole
`run_ours` path executes on the CPU (fp32, 2 steps) -- harness priming, the device-resident clip arm, the from-host clip arm,
the per-frame arms, the xcorr brackets, the JSON line.  Timings are meaningless here; the test pins the line's contract and
that the from-host clip arm tracks exactly what the device-resident arm tracked (bench.py refuses to report it otherwise)."""
import contextlib
import io
import json
import sys

import torch

import cabi_emulator


def test_bench_gpu_arm_control_flow_and_json_contract(monkeypatch, tmp_path):
    cabi_emulator.install_for_bench(monkeypatch)
    import bench
    from siammot_b200 import _lib, ops

    def xcorr_planar_any_dtype(x_planar, k, out=None, mma_mode=None):   # the emulation is fp32: lift the wrapper's fp16 requirement
        n, Cc, _ = x_planar.shape
        out = torch.empty((n, 16, 16, Cc), dtype=k.dtype) if out is None else out
        _lib.check(_lib.lib().smot_xcorr_planar(ops._ptr(x_planar), ops._ptr(k), ops._ptr(out), n, Cc, None))
        return out
    monkeypatch.setattr(ops, "xcorr_planar", xcorr_planar_any_dtype)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "3", "--dtype", "float32", "--no-cpu-baseline",
                                      "--experimental", "inproc", "--workload", "selftest", "--dump-outputs", str(tmp_path / "out")])
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            bench.main()
    finally:
        bench.select_workload("720p30")
    line = json.loads(buf.getvalue().strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
        assert key in line, key
    assert line["steps"] == 2 and line["n_gpus"] == 1 and line["config"]["tracks_in_memory"] == 8
    assert line["config"]["tracked_boxes_per_step"] >= 4          # tracks in memory are tracked (plus new detections)
    e2e = line["e2e"]
    assert e2e["clip_error"] is None and e2e["api"].startswith("model.forward_clip")
    assert e2e["h2d_bytes_per_step"] >= 3 * 256 * 384 and e2e["d2h_bytes_per_step"] > 0
    assert {"value", "unit"} <= set(e2e["per_frame_call"]) and {"value", "unit"} <= set(e2e["float32_chw_host_input"])
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["algorithmic_bytes"] == 8 * 128 * 1381 * 4 and 0 < r["frac"]
    assert line["gpu_launches"] > 0
    # --dump-outputs: the last timed step's result as float arrays of one box count, tracks in memory among the ids
    import numpy as np
    dump = {n: np.load(str(tmp_path / "out" / (n + ".npy"))) for n in ("boxes", "scores", "ids", "labels")}
    n = dump["boxes"].shape[0]
    assert dump["boxes"].shape == (n, 4) and n > 0 and all(dump[k].shape == (n,) for k in ("scores", "ids", "labels"))
    assert dump["boxes"].dtype == dump["scores"].dtype == np.float32 and dump["ids"].dtype == dump["labels"].dtype == np.float64
    assert int((dump["ids"] >= 0).sum()) >= 4
    # the information-only arms: three-stage clip (K = 2, 3) tracks what the two-stream clip tracks; the planar exchange
    # reproduces the default kernels' windows and responses
    ex = line["experimental"]
    for k in ("three_stage_clip_k2", "three_stage_clip_k3"):
        assert ex[k].get("same_tracks_as_two_stream") is True, ex[k]
    assert ex["xcorr_planar"].get("windows_equal_default") is True and ex["xcorr_planar"].get("output_equal_default") is True, ex["xcorr_planar"]
    for k in ("default_kernel", "mma_phase_of_default_kernel", "trimmed_mma_phase"):
        assert "us_per_launch" in ex["xcorr_planar"][k]["eager"] and "us_per_launch" in ex["xcorr_planar"][k]["graph"], ex["xcorr_planar"][k]


def test_bench_experimental_child_mode(monkeypatch):
    """`bench.py --experimental child` (what the default run launches as a subprocess once its own line is final)."""
    cabi_emulator.install_for_bench(monkeypatch)
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "2", "--warmup", "3", "--dtype", "float32", "--experimental", "child",
                                      "--workload", "selftest"])
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            bench.main()
    finally:
        bench.select_workload("720p30")
    ex = json.loads(buf.getvalue().strip().splitlines()[-1])
    assert ex["three_stage_clip_k2"]["same_tracks_as_two_stream"] is True and ex["three_stage_clip_k3"]["same_tracks_as_two_stream"] is True
    assert "xcorr_planar" in ex        # fp32 here: the wrapper refuses (TypeError recorded), fp16 on the GPU
    assert ex["frame_overlap"].get("same_tracks_as_default") is True, ex["frame_overlap"]


def test_demo_clip_tool_end_to_end(monkeypatch, tmp_path):
    """tools/demo_clip.py (the engine's demos/demo.py): raw frames -> forward_clip -> egress -> JSON, over the emulation."""
    import os
    cabi_emulator.install_for_bench(monkeypatch)
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import demo_clip
    out = tmp_path / "tracks.json"
    kept = demo_clip.main(["--synthetic", "6", "--size", "192x320", "--dtype", "float32", "--track-len", "2", "--track-conf", "0.0",
                           "--out", str(out)])
    recs = json.loads(out.read_text())
    assert len(recs) == len(kept) and all(set(r) == {"frame_num", "id", "label", "confidence", "bbox"} for r in recs)
    assert all(r["id"] >= 0 and len(r["bbox"]) == 4 for r in recs)
