"""bench.py's distributed branch (`--gpus N` under torchrun) on the CPU: two ranks, gloo, the C-ABI emulator, and -- the
combination that broke every N>1 run of round 1 -- `model.results_on_host = True` (CPU BoxLists) feeding the per-clip gather.

Two things are pinned:
  * the whole branch runs to the JSON line at world size 2 (rank 0 prints it, value aggregates both ranks, the gathered
    records of both ranks arrive);
  * under an NCCL process group no CPU tensor ever reaches a collective: the records are packed on the rank's CUDA device
    (checked with the backend reported as "nccl" and the packing intercepted -- there is no GPU in this container).
"""
import contextlib
import io
import json
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _bench_rank(rank, world, port, q):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), SMOT_BENCH_BACKEND="gloo")
    import cabi_emulator
    mpatch = pytest.MonkeyPatch()
    try:
        cabi_emulator.install_for_bench(mpatch)
        import bench
        mpatch.setattr(bench, "SETTLE_S", 0.0)
        mpatch.setattr(sys, "argv", ["bench.py", "--gpus", str(world), "--steps", "2", "--warmup", "3", "--dtype", "float32",
                                     "--no-cpu-baseline", "--experimental", "off", "--workload", "selftest"])
        import torch.distributed as dist
        seen = []
        orig_gather, orig_reduce = dist.all_gather, dist.all_reduce

        def spy_gather(parts, t, *a, **k):
            seen.append(("all_gather", t.device.type))
            return orig_gather(parts, t, *a, **k)

        def spy_reduce(t, *a, **k):
            seen.append(("all_reduce", t.device.type))
            return orig_reduce(t, *a, **k)
        mpatch.setattr(dist, "all_gather", spy_gather)
        mpatch.setattr(dist, "all_reduce", spy_reduce)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            bench.main()
        q.put((rank, buf.getvalue(), seen, None))
    except BaseException as exc:   # noqa: B902 -- report, never hang the parent
        import traceback
        q.put((rank, "", [], "%s\n%s" % (exc, traceback.format_exc())))
    finally:
        mpatch.undo()


def test_bench_distributed_branch_world2_results_on_host():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_bench_rank, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, out, seen, err in res:
        assert err is None, "rank %d: %s" % (rank, err)
        # gloo group: every tensor handed to a collective lives on the host (the exchange device of the backend)
        assert seen and all(dev == "cpu" for _, dev in seen), seen
        assert any(op == "all_gather" for op, _ in seen)
    assert res[1][1].strip() == ""                                   # only rank 0 prints
    line = json.loads(res[0][1].strip().splitlines()[-1])
    assert line["n_gpus"] == 2 and line["scaling"] == "weak" and line["steps"] == 2
    assert line["config"]["parallelism"].endswith("x 2")
    pr = line["per_rank_ms"]
    assert len(pr["rows"]) == 2 and len(pr["gathered_tracks_per_rank"]) == 2
    assert all(n > 0 for n in pr["gathered_tracks_per_rank"])        # both ranks' track states arrived
    assert line["e2e"]["clip_error"] is None
    # value is the whole-job aggregate: 2 ranks x 2 steps over the slowest rank's timed region
    assert abs(line["value"] - 2 * 2 / (line["ms_per_step"] * 2 * 1e-3)) / line["value"] < 1e-2


def test_records_are_packed_on_the_cuda_device_under_nccl(monkeypatch):
    """NCCL has no CPU backend: with results_on_host the BoxList is a CPU tensor, the records must not be."""
    import torch.distributed as dist
    sys.path.insert(0, REPO)
    from siammot_b200 import parallel
    from siammot_b200.structures import BoxList
    b = BoxList(torch.zeros((3, 4)), (1280, 704))
    b.add_field("scores", torch.ones(3))
    b.add_field("ids", torch.tensor([0, 1, -1]))
    b.add_field("labels", torch.ones(3, dtype=torch.int64))
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_backend", lambda group=None: "nccl")
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 3)
    assert parallel.exchange_device(b) == torch.device("cuda", 3)
    devices = []

    class Stop(Exception):
        pass

    def fake_pack(result, max_tracks, device=None):
        devices.append(device)
        raise Stop()
    monkeypatch.setattr(parallel, "pack_track_states", fake_pack)
    with pytest.raises(Stop):
        parallel.gather_track_states(b, max_tracks=8)
    assert devices == [torch.device("cuda", 3)]
    monkeypatch.setattr(dist, "get_backend", lambda group=None: "gloo")
    assert parallel.exchange_device(b) == torch.device("cpu")


def test_reference_arm_prints_the_same_config_keys(monkeypatch):
    """--impl reference under torchrun: rank 0 only, all host threads (torchrun's OMP_NUM_THREADS=1 overridden), the
    warm-up count honoured, `config` with the keys of our arm."""
    sys.path.insert(0, REPO)
    import bench
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--workload", "selftest"])
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.main()
    assert buf.getvalue() == ""                                        # other ranks exit 0 without work
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("WORLD_SIZE", "2")
    calls = []
    monkeypatch.setattr(bench, "oracle_runner", lambda: (lambda i: calls.append(i) or {"ids": torch.tensor([0, -1, 2])}))
    expected_threads = bench.host_threads()            # calibrated once (cached), before set_num_threads is intercepted
    threads = []
    monkeypatch.setattr(torch, "set_num_threads", lambda n: threads.append(n))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "2", "--workload", "selftest"])
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            bench.main()
        line = json.loads(buf.getvalue().strip().splitlines()[-1])
        ours = bench.config_dict(2)
    finally:
        bench.select_workload("720p30")
    assert calls == [0, 1, 2, 3, 4] and line["warmup"] == 2 and line["steps"] == 3
    assert threads and threads[0] == expected_threads >= 1
    assert line["impl"] == "reference" and line["cpu_baseline"]["cores"] == threads[0]
    assert set(line["config"]) == set(ours) | {"tracked_boxes_per_step"}
    assert {k: line["config"][k] for k in ours} == ours
    assert line["config"]["tracked_boxes_per_step"] == 2.0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
