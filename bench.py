#!/usr/bin/env python
"""bench.py -- SiamMOT hot-path throughput on B200 (contract: see the task statement / DESIGN.md).

A "step" is one frame through the per-frame hot path (backbone -> FPN -> RPN -> box head -> EMM with
30 tracks in memory -> refinement -> solver -> next-frame memory) on the BASELINE.json configs[1]
workload: 1280x720 synthetic video, i.e. a 3x704x1280 network input after the reference's own resize
rule (image_augmentation.py:21-42), DLA-34-FPN + EMM, fp16 storage / fp32 accumulation.
`value`: model.forward_clip over normalised frames resident in HBM; `e2e`: model.forward_clip over decoded uint8 frames in
pinned host memory (per frame: H2D, test transform on the device, hot path, packed result D2H -- all inside the wall-clock
region); `e2e.per_frame_call`: the same frames through model(frame), one blocking call per frame.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype float16|float32] [--dump-outputs DIR]
  python bench.py --impl reference ...     # the reference path on the host CPU (oracle port)
  torchrun --nproc-per-node N bench.py --gpus N ...   # one process per GPU, independent streams

Each arm times exactly K steps.  Prints ONE JSON line on rank 0.  --dump-outputs DIR writes what the timed path returned for its
last step as DIR/<name>.npy (see dump_outputs); the inputs are a pure function of the arguments, so two builds can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True    # the tree may be read-only, and a benchmark run leaves it as it found it

import torch  # noqa: E402

H_NET, W_NET = 704, 1280      # 1280x720 after the reference's test-time resize (SURVEY.md fact 5)
H_SRC, W_SRC = 720, 1280      # the decoded video frame (RGB uint8)
N_TRACKS = 30
N_FRAMES = 32                 # distinct frames resident in HBM: 32 x 10.8 MB = 346 MB > 126 MB L2
METRIC = "tracker FPS @720p (DLA34-FPN+EMM, 30 tracks)"
WORKLOAD = "720p synthetic clip -> 3x704x1280, DLA-34-FPN + EMM, 30 active tracks, 1 frame per step"
CFG_OVERRIDES = []
CFG_YAML = "dla34_emm.yaml"

# BASELINE.json configs: the default (configs[1]) is what the metric is quoted on; the others are selectable for reporting
WORKLOADS = {
    "720p30": dict(src=(720, 1280), net=(704, 1280), tracks=30, opts=[], yaml="dla34_emm.yaml",
                   metric=METRIC, text=WORKLOAD),
    # configs[4]: the same clip on the upstream R-50-FPN body (256-channel FPN / RPN / box head / EMM)
    "r50_720p30": dict(src=(720, 1280), net=(704, 1280), tracks=30, opts=[], yaml="r50_emm.yaml",
                       metric="tracker FPS @720p (R50-FPN+EMM, 30 tracks)",
                       text="720p synthetic clip -> 3x704x1280, R-50-FPN + EMM (256 channels), 30 active tracks, 1 frame per step"),
    # configs[2]: native 1080p input (INPUT.MIN/MAX_SIZE_TEST 1080/1920 -> 3x1056x1920, SURVEY.md 8d config 3), 80 tracks
    "1080p80": dict(src=(1080, 1920), net=(1056, 1920), tracks=80, opts=["INPUT.MIN_SIZE_TEST", 1080, "INPUT.MAX_SIZE_TEST", 1920],
                    yaml="dla34_emm.yaml",
                    metric="tracker FPS @1080p (DLA34-FPN+EMM, 80 tracks)",
                    text="1080p synthetic clip -> 3x1056x1920, DLA-34-FPN + EMM (search region r=2), 80 active tracks, 1 frame per step"),
    # not a benchmark: a small frame for tests/test_bench_emulated_cpu.py, which runs this file's control flow on the CPU
    "selftest": dict(src=(256, 384), net=(256, 384), tracks=8, opts=["INPUT.MIN_SIZE_TEST", 256, "INPUT.MAX_SIZE_TEST", 384],
                     yaml="dla34_emm.yaml", metric="(self-test, not a measurement)",
                     text="self-test clip -> 3x256x384, DLA-34-FPN + EMM, 8 active tracks, 1 frame per step"),
}


def select_workload(name):
    global H_NET, W_NET, H_SRC, W_SRC, N_TRACKS, METRIC, WORKLOAD, CFG_OVERRIDES, CFG_YAML
    w = WORKLOADS[name]
    CFG_YAML = w["yaml"]
    (H_SRC, W_SRC), (H_NET, W_NET), N_TRACKS = w["src"], w["net"], w["tracks"]
    METRIC, WORKLOAD, CFG_OVERRIDES = w["metric"], w["text"], w["opts"]


def config_dict(world=1):
    """The `config` object of the JSON line: identical for both arms (ours / --impl reference), so the driver compares like with
    like.  Arm-specific notes (API used, graphs, baseline note) live in `notes`, outside it."""
    return {"workload": WORKLOAD, "net_input": [3, H_NET, W_NET], "source_frame": [H_SRC, W_SRC, 3], "frames_resident": N_FRAMES,
            "l2": "inputs (%d MB of frames + activations) exceed the 126 MB L2" % (N_FRAMES * 3 * H_NET * W_NET * 4 // 1000000),
            "tracks_in_memory": N_TRACKS, "parallelism": "1 stream per GPU x %d" % world}


_HOST_THREADS = None


def host_threads():
    """The torch thread count that makes the CPU legs fastest on this host, found by timing a small convolution at
    4 / 8 / 16 / ... / all CPUs this process may use (bounded by the cgroup CPU quota when there is one).  "All the host
    threads it can use" is not the affinity count on a shared box: on the round-2 GPU hosts 128 threads made the oracle 40x
    SLOWER than 8 (quota + hyper-threads), which would have flattered the GPU/CPU ratio.  torchrun's OMP_NUM_THREADS=1 is
    overridden by whoever calls torch.set_num_threads(host_threads())."""
    global _HOST_THREADS
    if _HOST_THREADS is not None:
        return _HOST_THREADS
    try:
        limit = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        limit = max(1, os.cpu_count() or 1)
    try:   # cgroup v2 / v1 CPU quota
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            limit = max(1, min(limit, int(float(q[0]) / float(q[1]) + 0.5)))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                limit = max(1, min(limit, (quota + period // 2) // period))
        except Exception:
            pass
    cands = sorted({c for c in (4, 8, 16, 32, 64, 128, 256) if c < limit} | {limit})
    keep = torch.get_num_threads()
    # two layers of the path's mix (a level-2 and a level-4 conv); per candidate the MINIMUM of 5 trials, so that a neighbour's
    # burst on a shared host does not pick the thread count (one noisy trial once chose 4 threads where 16 are 1.6x faster)
    shapes = [(torch.randn(1, 64, 176, 320), torch.randn(64, 64, 3, 3)), (torch.randn(1, 256, 44, 80), torch.randn(256, 256, 3, 3))]
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        for x, w in shapes:
            torch.nn.functional.conv2d(x, w, padding=1)
        dt = float("inf")
        for _ in range(5):
            t0 = time.perf_counter()
            for x, w in shapes:
                torch.nn.functional.conv2d(x, w, padding=1)
            dt = min(dt, time.perf_counter() - t0)
        if dt < 0.95 * best_t:       # prefer fewer threads unless clearly faster
            best, best_t = c, dt
    torch.set_num_threads(keep)
    _HOST_THREADS = best
    return best


def pin_to_gpu_numa_node(local):
    """Bind this rank to the CPUs NVML reports as local to its GPU (on the 8-GPU box GPUs 0-3 sit on one socket, 4-7 on the
    other): the host solver, the pinned staging buffers and the launch loop then stay on the GPU's own NUMA node.
    Returns the number of CPUs bound, or None when NVML / the affinity call is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def build_cfg(dtype):
    from siammot_b200.config import get_cfg
    cfg = get_cfg()
    cfg.merge_from_file(os.path.join(REPO, "siammot_b200", "configs", CFG_YAML))
    if CFG_OVERRIDES:
        cfg.merge_from_list(list(CFG_OVERRIDES))
    cfg.DTYPE = dtype
    return cfg


def track_table(n=None):
    """N_TRACKS pedestrian-like boxes spread over the frame (cx, cy, w, h), hitting FPN levels 0..2."""
    n = N_TRACKS if n is None else n
    if (H_NET, W_NET) == (256, 384):      # the self-test frame: the 720p table scaled down
        return _track_table_720p(n) * torch.tensor([384 / 1280., 256 / 704., 384 / 1280., 256 / 704.])
    return _track_table_720p(n)


def _track_table_720p(n):
    g = torch.Generator().manual_seed(123)
    W, H = (1280, 704) if (H_NET, W_NET) == (256, 384) else (W_NET, H_NET)
    cx = torch.rand(n, generator=g) * (W - 200) + 100
    cy = torch.rand(n, generator=g) * (H - 300) + 150
    h = torch.rand(n, generator=g) * 260 + 60
    w = h * (0.3 + 0.2 * torch.rand(n, generator=g))
    return torch.stack((cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2), dim=1)


def make_frames_u8(n, cfg):
    """Decoded 720p RGB uint8 frames (n, 720, 1280, 3): what a video reader hands to the tracker."""
    from siammot_b200.synth_clip import make_clip_u8
    return make_clip_u8(n, H_SRC, W_SRC, n_obj=12, seed=0, mean=cfg.INPUT.PIXEL_MEAN, std=cfg.INPUT.PIXEL_STD)


# --------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
class Harness(object):
    """Owns the model and restores the fixed 30-track memory before every step, so each step is one
    natural frame with exactly 30 tracks (all active) in memory."""

    def __init__(self, dtype, device):
        from siammot_b200.modelling import build_siammot
        from siammot_b200.synthetic import make_state_dict
        self.cfg = build_cfg(dtype)
        self.model = build_siammot(self.cfg)
        self.model.load_state_dict(make_state_dict(self.cfg, 1), strict=False)
        self.model = self.model.to(device).eval()
        self.device = device
        self.eng = self.model.engine()
        self.pool = self.model.roi_heads.track.track_pool
        self.boxes = track_table()
        self.mem = None

    def prime(self, frame_dev):
        P = self.eng.run_static(frame_dev)
        self.pool.reset()
        ids = torch.tensor([self.pool.start_track() for _ in range(N_TRACKS)])
        self.mem = self.model.roi_heads._build_memory(P, self.boxes.numpy(), ids.numpy(),
                                                      torch.ones(N_TRACKS, dtype=torch.int64).numpy())
        self.pool.increment_frame()
        self.snapshot = (set(self.pool._active_ids), dict(self.pool._dormant_ids), dict(self.pool._cache),
                         self.pool._max_id, self.pool._frame_idx)

    def restore(self):
        a, d, c, m, f = self.snapshot
        p = self.pool
        p._active_ids, p._dormant_ids, p._cache, p._max_id, p._frame_idx = set(a), dict(d), dict(c), m, f
        self.model.flush_memory(self.mem)

    def step(self, frame):
        self.restore()
        return self.model(frame)[0]


def kernels_per_frame(h):
    """Kernels of libsmot.so launched per step: static plan (graph replay) + dynamic stage at N=30."""
    from siammot_b200 import _lib
    P = h.eng.plan(H_NET, W_NET)
    n = 0
    for fn, args, tag, _branch in P.steps:
        name = getattr(fn, "__name__", None)
        n += _lib.KERNELS_PER_CALL.get(name, 0) if name else 0
    # dynamic: sr roi_align, xcorr, towers conv, groupnorm, 2 head convs, decode(2), refine(roi_align, 3 conv, decode),
    # solver sort_nms, template roi_align
    n += 1 + 1 + 1 + 1 + 2 + 2 + 5 + 1 + 3 + 1
    return n


SETTLE_S = 0.4   # untimed repeats of an arm's region before its timed one


def settle(run):
    """Run the arm's K-step region untimed, at least twice and for SETTLE_S: right after set-up the first region runs slow (on a
    B200 the first of twenty 20-step regions ran at 72 % of the median of the others), and one timed region of K steps must
    not measure that ramp."""
    t0, n = time.perf_counter(), 0
    while n < 2 or time.perf_counter() - t0 < SETTLE_S:
        run()
        torch.cuda.synchronize()
        n += 1


def dump_outputs(path, boxes, scores, ids, labels):
    """What a caller of the timed path receives for its last step, as DIR/<name>.npy: boxes (N x 4, xyxy in network-input
    pixels) and scores as float32, track ids (-1: a detection no track claimed) and class labels as float64 (exact)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in (("boxes", boxes), ("scores", scores), ("ids", ids), ("labels", labels)):
        a = t.detach().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64 if a.dtype.kind in "iub" else np.float32))


def run_ours(args):
    distributed = args.gpus > 1 and "RANK" in os.environ
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1)) if distributed else 1
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    numa_cpus = pin_to_gpu_numa_node(local) if distributed else None
    if distributed:
        import torch.distributed as dist
        # SMOT_BENCH_BACKEND=gloo: the CPU test of this branch (tests/test_bench_distributed_cpu.py); production is NCCL
        backend = os.environ.get("SMOT_BENCH_BACKEND", "nccl")
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=device)
        else:
            dist.init_process_group(backend)
        from siammot_b200.parallel import exchange_device
        xdev = exchange_device()           # where tensors handed to a collective must live (the rank's GPU under NCCL)
    torch.set_num_threads(max(1, min(8, host_threads() // max(world, 1))))   # the host side is one Python thread + small numpy ops
    h = Harness(args.dtype, device)
    h.model.results_on_host = True   # results are consumed on the host (as demo / inferencer do): CPU BoxLists straight from the solver
    frames_u8 = make_frames_u8(N_FRAMES, h.cfg).pin_memory()                   # host, pinned: the e2e arm's input
    pre = h.eng.preprocessor()
    frames_dev = torch.stack([pre(frames_u8[i]) for i in range(N_FRAMES)])    # normalised 3x704x1280, resident in HBM
    frames_pin = frames_dev.cpu().pin_memory()                                 # the reference-style float input (host)
    assert tuple(frames_dev.shape[1:]) == (3, H_NET, W_NET)
    h.prime(frames_dev[0])

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: `value` (clip API: the detection stage of frame t+1 overlaps the host solver of frame t).
    # No event timers in this arm (they are on only in the per-frame arm below); one timed region of exactly K steps.
    hook = lambda t: h.restore()
    h.eng.timers = None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    h.model.forward_clip([frames_dev[i % N_FRAMES] for i in range(max(args.warmup, 4))], before_frame=hook)
    seq = [frames_dev[(args.warmup + i) % N_FRAMES] for i in range(args.steps)]
    settle(lambda: h.model.forward_clip(seq, before_frame=hook))
    barrier()
    h.eng.host_timers = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    results = h.model.forward_clip(seq, before_frame=hook)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    host_t, h.eng.host_timers = h.eng.host_timers, None
    ntrk = sum(int((r.get_field("ids") >= 0).sum()) for r in results)
    r = results[-1]

    # ---- end-to-end arm through the public API with HOST frames: `e2e`.  The call a user makes per decoded frame:
    # model(uint8 HWC frame) -> H2D of the frame, test transform on the device, the whole hot path, D2H of the result.
    def e2e_loop(src):
        for i in range(min(args.warmup, 3)):
            h.step(src[i % N_FRAMES]).to("cpu")
        barrier()
        t0 = time.perf_counter()
        nbytes = 0
        for i in range(args.steps):
            h.restore()
            out = h.model(src[(args.warmup + i) % N_FRAMES])[0].to("cpu")   # H2D inside forward; results arrive on the host
            nbytes += out.bbox.numel() * 4 + sum(out.get_field(f).numel() * out.get_field(f).element_size() for f in out.fields())
        torch.cuda.synchronize()
        return time.perf_counter() - t0, nbytes

    # The same from-host measurement through the clip API (the call a user makes for a decoded video: all frames of the
    # clip are on the host, pinned): per frame, the uint8 frame's H2D copy + test transform + detection stage run on the side
    # stream while the previous frame's track stage / host solver run; results arrive as CPU BoxLists (packed block D2H).
    def e2e_clip_loop(src):
        h.model.forward_clip([src[i % N_FRAMES] for i in range(max(args.warmup, 4))], before_frame=hook)
        seq_h = [src[(args.warmup + i) % N_FRAMES] for i in range(args.steps)]
        settle(lambda: h.model.forward_clip(seq_h, before_frame=hook))
        barrier()
        t0 = time.perf_counter()
        res = h.model.forward_clip(seq_h, before_frame=hook)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert len(res) == args.steps and all(r.bbox.device.type == "cpu" for r in res)
        return dt, sum(int((r.get_field("ids") >= 0).sum()) for r in res)

    e2e_clip_s, e2e_clip_err = None, None
    try:
        e2e_clip_s, ntrk_clip = e2e_clip_loop(frames_u8)
        if ntrk_clip != ntrk:   # same frames, same restored memory: the from-host clip must track exactly what `value` tracked
            e2e_clip_err = "clip-from-host tracked %d boxes, device-resident clip %d" % (ntrk_clip, ntrk)
    except Exception as exc:   # keep the per-frame number as the headline rather than lose the line
        e2e_clip_err = "%s: %s" % (type(exc).__name__, exc)
        torch.cuda.synchronize()

    # per-kernel CUDA-event brackets are taken in this arm: its launches are on ONE stream, so a bracket times the
    # kernel alone (in the clip arm the other stream's kernels run inside the bracket)
    h.eng.timers = {}
    e2e_s, d2h = e2e_loop(frames_u8)
    timers, h.eng.timers = h.eng.timers, None
    static = [a.elapsed_time(b) for a, b in timers.get("static", [])][min(args.warmup, 3):]
    prep = [a.elapsed_time(b) for a, b in timers.get("preprocess", [])][min(args.warmup, 3):]
    e2e_float_s, _ = e2e_loop(frames_pin)   # the reference's calling convention: normalised float32 CHW host tensor
    clocks = sampler.stop() if rank == 0 else None   # sampled across both timed arms
    # roofline kernel: the frame's own correlation launch (same buffers: the search windows / templates of the last frame,
    # L2-resident as in the pipeline), bracketed with CUDA events on its stream, right after the timed region.  Measured both
    # ways: eagerly (20 back-to-back launches from the Python/ctypes loop) and as a 20-launch CUDA-graph replay, which is how
    # the product issues it (the track stage is a graph; a ~4 us kernel launched eagerly is paced by the ~8 us launch loop).
    from siammot_b200._lib import check, stream_ptr
    tp = h.eng.track_plan(h.eng.plan(H_NET, W_NET), N_TRACKS)
    xfn, xargs, _ = tp.steps[tp.xcorr_slot]
    xc_t = time_launches(lambda: check(xfn(*xargs, stream_ptr()), "xcorr"))

    clip_ok = e2e_clip_s is not None and e2e_clip_err is None
    static_ms = sum(static) / max(len(static), 1)
    prep_ms = sum(prep) / max(len(prep), 1)
    per_rank = None
    if distributed:
        t = torch.tensor([ms, e2e_s * 1e3, e2e_float_s * 1e3, e2e_clip_s * 1e3 if clip_ok else float("inf"), static_ms, prep_ms],
                         device=xdev, dtype=torch.float64)
        allr = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allr, t)
        per_rank = [[round(float(v), 4) for v in x.tolist()] for x in allr]
        t = torch.stack(allr).max(dim=0).values      # MAX over ranks of every time
        ms, e2e_ms, e2e_float_ms, e2e_clip_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        clip_ok = e2e_clip_ms != float("inf")   # every rank's clip arm ran
        # the one inference collective: per-clip gather of fixed-size track-state records (SURVEY.md 8e), on the exchange device
        from siammot_b200.parallel import gather_track_states, unpack_track_states
        rec = gather_track_states(r, max_tracks=128)
        assert rec.shape[0] == world and rec.device.type == xdev.type, (rec.shape, rec.device)
        gathered = [int(s_["ids"].numel()) for s_ in unpack_track_states(rec.cpu())]
    else:
        e2e_ms, e2e_float_ms = e2e_s * 1e3, e2e_float_s * 1e3
        e2e_clip_ms = e2e_clip_s * 1e3 if clip_ok else float("inf")
        gathered = None
    if rank != 0:
        if distributed:
            dist.barrier()
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    esz = 2 if args.dtype == "float16" else 4
    S_, T_ = h.eng.s_res, h.eng.t_res
    xc_bytes = N_TRACKS * h.eng.C * (S_ * S_ + T_ * T_ + (S_ - T_ + 1) ** 2) * esz      # SURVEY.md 8(d): N*C*1381*b at S=30, T=15
    xc_best = xc_t.get("graph") if "us_per_launch" in xc_t.get("graph", {}) else xc_t.get("eager", {})
    xc_us = xc_best.get("us_per_launch", 0.0)
    achieved = xc_bytes / (xc_us * 1e-6) / 1e9 if xc_us > 0 else 0.0
    traffic = None
    try:
        # per launch, from one `ncu --set full` capture of the named kernel at this (tracks x channels); null when none is committed
        table = json.load(open(os.path.join(REPO, "profiles", "xcorr_traffic.json")))
        traffic = table.get(getattr(tp, "xcorr_kernel", "").split("<")[0].split(" ")[0], {}).get("%dx%d" % (N_TRACKS, h.eng.C))
    except Exception:
        pass
    fps = world * args.steps / (ms * 1e-3)
    e2e_fps = world * args.steps / ((e2e_clip_ms if clip_ok else e2e_ms) * 1e-3)
    cfgd = config_dict(world)
    cfgd["tracked_boxes_per_step"] = round(ntrk / args.steps, 1)
    out = {
        "metric": METRIC, "value": round(fps, 2), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": round(fps / world / 17.0, 2) if (world == 1 and args.workload == "720p30") else None,
        "dtype": "f16" if args.dtype == "float16" else "f32", "data": "synthetic",
        "config": cfgd,
        "notes": {"cuda_graph": True, "pipeline": h.eng.clip_mode_name(),
                  "api": "value: model.forward_clip on normalised frames resident in HBM; e2e: the same clip API on decoded RGB uint8 "
                         "720p frames in pinned host memory (per frame: 2.76 MB H2D + test transform resize 720->704 / ToTensor / "
                         "Normalize on the device, packed result block D2H; all inside the wall-clock region); "
                         "e2e.per_frame_call: model(frame) once per frame; "
                         "model.results_on_host = True (CPU BoxLists from the packed result block the engine copies D2H)",
                  "baseline_note": "17 FPS = README.md:22 'a single modern GPU', unnamed hardware",
                  "timed_steps": "one timed region of exactly %d steps per arm, after untimed repeats of it for >= %.1f s "
                                 "(max over ranks); e2e may exceed value by a few per cent: the device-resident arm reads 10.8 MB "
                                 "fp32 frames from HBM (image_to_nhwc), the host arm uploads 2.8 MB uint8 frames and resamples on the "
                                 "side stream" % (args.steps, SETTLE_S),
                  "numa_cpus_bound": numa_cpus},
        "e2e": {"value": round(e2e_fps, 2), "unit": "frames/s",
                "api": "model.forward_clip(pinned uint8 host frames)" if clip_ok else "model(pinned uint8 host frame) per frame",
                "h2d_bytes_per_step": 3 * H_SRC * W_SRC + tp.inputs.numel() * 4,
                "d2h_bytes_per_step": (tp.host_res.numel() + tp.host_det.numel()) * 4,
                "result_bytes_per_step": int(d2h / args.steps),
                "per_frame_call": {"value": round(world * args.steps / (e2e_ms * 1e-3), 2), "unit": "frames/s",
                                   "note": "model(frame) called once per decoded frame (demo.py's loop, the reference's own API)"},
                "clip_error": e2e_clip_err,
                "float32_chw_host_input": {"value": round(world * args.steps / (e2e_float_ms * 1e-3), 2), "unit": "frames/s",
                                           "h2d_bytes_per_step": 3 * H_NET * W_NET * 4,
                                           "note": "same per-frame loop with the reference's calling convention (frame already resized + "
                                                   "normalised on the host)"}},
        "gpu_launches": kernels_per_frame(h) * args.steps,
        "roofline": {"kernel": getattr(tp, "xcorr_kernel", "smot_xcorr"), "bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak,
                     "unit": "GB/s", "frac": round(achieved / hbm_peak, 4), "traffic": traffic,
                     "algorithmic_bytes": xc_bytes, "us_per_launch": round(xc_us, 2),
                     "us_per_launch_eager": xc_t.get("eager", {}).get("us_per_launch"),
                     "us_per_launch_graph": xc_t.get("graph", {}).get("us_per_launch"),
                     "timing": "10 CUDA-event brackets (after 3 warm-up ones) of 20 back-to-back launches of the frame's own correlation "
                               "call on its buffers, right after the timed region; `us_per_launch` is the CUDA-graph replay of the 20 "
                               "launches (the product issues the track stage as a graph), `us_per_launch_eager` the ctypes launch loop",
                     "peak_source": "MEASURED_PEAKS.json (burst copy)" if peaks else "fallback 6650 GB/s",
                     "flops_per_launch": N_TRACKS * h.eng.C * 2 * (S_ - T_ + 1) ** 2 * T_ * T_,
                     "note": getattr(tp, "xcorr_note", "")},
        "stage_ms": {"static_graph": round(static_ms, 4), "preprocess_incl_h2d": round(prep_ms, 4),
                     "note": "CUDA-event brackets in the per-frame e2e arm (single stream)",
                     "host_per_frame_ms": {k: round(v / max(host_t.get("frames", 1), 1) * 1e3, 4) for k, v in host_t.items() if k != "frames"},
                     "host_note": "wall clock inside finish_frame during the `value` arm: track_wait = blocking on the track "
                                  "stage's result block (its GPU latency under the overlapped backbone), solver = unpack + id "
                                  "resolution, next_memory = staging + template pooling launch, boxlist = result object; their "
                                  "sum + the launch code is the sequential chain of a video"},
        "clocks": clocks,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r.bbox, r.get_field("scores"), r.get_field("ids"), r.get_field("labels"))
    if per_rank is not None:
        out["per_rank_ms"] = {"columns": ["value_region", "per_frame_region", "float_region", "e2e_clip_region", "static_graph", "preprocess"],
                              "rows": per_rank, "gathered_tracks_per_rank": gathered}
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(sample_frames=2)
    if world == 1 and args.experimental == "subprocess":
        # Paths that are built and host-verified but have not been through a GPU run yet (DESIGN.md 4 / 5.2) are measured for
        # information in a CHILD process after everything above is final: a crash, a CUDA error or a hang there cannot cost
        # the line (the child is killed at the timeout).
        out["experimental"] = experimental_subprocess(args)
    elif world == 1 and args.experimental == "inproc":
        def bail():
            out["experimental"] = {"error": "watchdog: the experimental arms did not return within %d s" % EXPERIMENTAL_TIMEOUT_S}
            print(json.dumps(out))
            sys.stdout.flush()
            os._exit(0)
        dog = threading.Timer(EXPERIMENTAL_TIMEOUT_S, bail)
        dog.daemon = True
        dog.start()
        try:
            out["experimental"] = experimental_arms(h, args, frames_dev, frames_u8, hook, ntrk, tp, hbm_peak, xc_bytes)
        except BaseException as exc:   # noqa: B902 -- a CUDA error surfaces as RuntimeError; keep the line whatever it is
            out["experimental"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
        dog.cancel()
    print(json.dumps(out))
    sys.stdout.flush()
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


EXPERIMENTAL_TIMEOUT_S = 150


def time_launches(launch, reps=20):
    """us per launch of `launch()` (one kernel on the current stream): CUDA-event brackets around `reps` back-to-back launches,
    10 brackets after 3 warm-up ones; 'eager' = the Python/ctypes launch loop, 'graph' = the launches replayed as one CUDA graph."""
    out = {}
    for how in ("eager", "graph"):
        try:
            if how == "graph":
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    launch()                         # function attributes are set outside the capture
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for _ in range(reps):
                        launch()
                run = g.replay
            else:
                def run():
                    for _ in range(reps):
                        launch()
            ev = []
            for i in range(13):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                run()
                b.record()
                ev.append((a, b))
            torch.cuda.synchronize()
            ms = sum(a.elapsed_time(b) / reps for a, b in ev[3:]) / max(len(ev) - 3, 1)
            out[how] = {"us_per_launch": round(ms * 1e3, 2)}
        except Exception as exc:
            out[how] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    return out


def experimental_subprocess(args):
    cmd = [sys.executable, os.path.abspath(__file__), "--experimental", "child", "--steps", str(args.steps), "--warmup", str(args.warmup),
           "--dtype", args.dtype, "--workload", args.workload]
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=EXPERIMENTAL_TIMEOUT_S)
    except subprocess.TimeoutExpired:
        return {"error": "child process killed after %d s" % EXPERIMENTAL_TIMEOUT_S}
    except Exception as exc:
        return {"error": "%s: %s" % (type(exc).__name__, exc)}
    for line in reversed(r.stdout.strip().splitlines()):
        try:
            return json.loads(line)
        except ValueError:
            continue
    return {"error": "child exited with code %d: %s" % (r.returncode, r.stderr.strip()[-300:])}


def run_experimental_child(args):
    """`bench.py --experimental child`: own process, own model; prints one JSON object (the "experimental" entry)."""
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    h = Harness(args.dtype, device)
    h.model.results_on_host = True
    frames_u8 = make_frames_u8(N_FRAMES, h.cfg).pin_memory()
    pre = h.eng.preprocessor()
    frames_dev = torch.stack([pre(frames_u8[i]) for i in range(N_FRAMES)])
    h.prime(frames_dev[0])
    hook = lambda t: h.restore()
    h.model.forward_clip([frames_dev[i % N_FRAMES] for i in range(max(args.warmup, 4))], before_frame=hook)
    torch.cuda.synchronize()
    tp = h.eng.track_plan(h.eng.plan(H_NET, W_NET), N_TRACKS)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    esz = 2 if args.dtype == "float16" else 4
    xc_bytes = N_TRACKS * h.eng.C * (30 * 30 + 15 * 15 + 16 * 16) * esz
    print(json.dumps(experimental_arms(h, args, frames_dev, frames_u8, hook, None, tp, float(peaks.get("hbm_gbs", 6650.0)), xc_bytes)))


def experimental_arms(h, args, frames_dev, frames_u8, hook, ntrk_ref, tp, hbm_peak, xc_bytes):
    """Measured for information only; none of this feeds `value` / `e2e` / `roofline`.
    (1) forward_clip as a three-stage pipeline (Engine.clip_split, K = 2 and 3 plan copies): same clip, same memory, must track
        exactly the boxes the two-stream pipeline tracked.
    (2) the channel-planar search-window exchange: smot_roi_align_planar / smot_xcorr_planar on the last frame's own track
        inputs, compared bit for bit with the default kernels' outputs, then timed like the roofline kernel."""
    from siammot_b200 import _lib, ops
    from siammot_b200._lib import check, stream_ptr
    eng = h.eng
    res = {}
    steps = min(args.steps, 100)
    seq = [frames_dev[(args.warmup + i) % N_FRAMES] for i in range(steps)]
    seq_h = [frames_u8[(args.warmup + i) % N_FRAMES] for i in range(steps)]
    ref_trk = None
    for K in (2, 3):
        key = "three_stage_clip_k%d" % K
        try:
            eng.clip_split, eng.clip_slots = True, K
            h.model.forward_clip([frames_dev[i % N_FRAMES] for i in range(max(args.warmup, 4))], before_frame=hook)
            torch.cuda.synchronize()
            if ref_trk is None:   # the two-stream pipeline on exactly this (possibly shorter) sequence
                eng.clip_split = False
                ref_trk = sum(int((r.get_field("ids") >= 0).sum()) for r in h.model.forward_clip(seq, before_frame=hook))
                eng.clip_split = True
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = h.model.forward_clip(seq, before_frame=hook)
            e1.record()
            torch.cuda.synchronize()
            n1 = sum(int((r.get_field("ids") >= 0).sum()) for r in out)
            h.model.forward_clip(seq_h[:4], before_frame=hook)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = h.model.forward_clip(seq_h, before_frame=hook)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            n2 = sum(int((r.get_field("ids") >= 0).sum()) for r in out)
            res[key] = {"value": round(steps / (e0.elapsed_time(e1) * 1e-3), 2), "e2e": round(steps / dt, 2), "unit": "frames/s",
                        "steps": steps, "same_tracks_as_two_stream": bool(n1 == ref_trk and n2 == ref_trk)}
        except Exception as exc:
            res[key] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            break
        finally:
            eng.clip_split, eng.clip_slots = False, 2
    try:   # (3) model(frame) with the detection tail under the EMM half of the track stage (Engine.frame_overlap)
        def per_frame(flag):
            eng.frame_overlap = flag
            for i in range(3):
                h.step(frames_u8[i % N_FRAMES])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = 0
            for i in range(steps):
                n += int((h.step(frames_u8[(args.warmup + i) % N_FRAMES]).get_field("ids") >= 0).sum())
            torch.cuda.synchronize()
            return steps / (time.perf_counter() - t0), n
        fps0, n0 = per_frame(False)
        fps1, n1 = per_frame(True)
        fps1, n1 = per_frame(True)          # second pass: the per-half CUDA graphs exist
        res["frame_overlap"] = {"per_frame_call": round(fps1, 2), "per_frame_call_default": round(fps0, 2), "unit": "frames/s",
                                "steps": steps, "same_tracks_as_default": bool(n0 == n1)}
    except Exception as exc:
        res["frame_overlap"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    finally:
        eng.frame_overlap = False
    try:
        T = h.cfg.MODEL.TRACK_HEAD
        P = tp.P
        if eng.s_res != 30 or eng.t_res != 15:
            raise RuntimeError("planar exchange: S=30, T=15 only")
        srf = ops.roi_align(P.feats, tp.sr, T.POOLER_SCALES, eng.s_res, T.POOLER_SAMPLING_RATIO, level_boxes=tp.boxes, pads=eng.pads)
        srp = ops.roi_align_planar(P.feats, tp.sr, T.POOLER_SCALES, eng.s_res, T.POOLER_SAMPLING_RATIO, level_boxes=tp.boxes,
                                   pads=eng.pads)
        n, Cc = srf.shape[0], srf.shape[3]
        rows = srp[:, :, :30 * _lib.XCORR_ROW_PITCH].reshape(n, Cc, 30, _lib.XCORR_ROW_PITCH)
        same_windows = bool(torch.equal(rows[..., :30].permute(0, 2, 3, 1), srf)) and float(rows[..., 30:32].abs().max()) == 0.0
        tmpl = tp.tmpl.contiguous()
        ref = ops.xcorr(srf, tmpl)
        got = ops.xcorr_planar(srp, tmpl)
        same_out = bool(torch.equal(ref, got))
        L = _lib.lib()
        res["xcorr_planar"] = {"windows_equal_default": same_windows, "output_equal_default": same_out, "algorithmic_bytes": xc_bytes,
                               "timing": "20 launches per CUDA-event bracket, 10 brackets after 3 warm-up ones; 'graph': the 20 launches "
                                         "replayed as one CUDA graph (a ~4 us kernel is otherwise paced by the ~8 us Python/ctypes "
                                         "launch loop, which is also what times the default kernel in `roofline`)"}

        def time_launches(launch):
            out = {}
            for how in ("eager", "graph"):
                try:
                    if how == "graph":
                        side = torch.cuda.Stream()
                        side.wait_stream(torch.cuda.current_stream())
                        with torch.cuda.stream(side):
                            launch()                         # function attributes are set outside the capture
                        torch.cuda.current_stream().wait_stream(side)
                        torch.cuda.synchronize()
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g):
                            for _ in range(20):
                                launch()
                        run = g.replay
                    else:
                        def run():
                            for _ in range(20):
                                launch()
                    ev = []
                    for i in range(13):
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        run()
                        b.record()
                        ev.append((a, b))
                    torch.cuda.synchronize()
                    ms = sum(a.elapsed_time(b) / 20 for a, b in ev[3:]) / max(len(ev) - 3, 1)
                    gbs = xc_bytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
                    out[how] = {"us_per_launch": round(ms * 1e3, 2), "achieved_gbs": round(gbs, 1), "frac": round(gbs / hbm_peak, 4)}
                except Exception as exc:
                    out[how] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            return out

        dflt = torch.empty_like(ref)
        res["xcorr_planar"]["default_kernel"] = time_launches(
            lambda: check(L.smot_xcorr(ops._ptr(srf), ops._ptr(tmpl), ops._ptr(dflt), n, Cc, 30, 15, _lib.F16, stream_ptr()), "xcorr"))
        for mode, key in ((0, "mma_phase_of_default_kernel"), (1, "trimmed_mma_phase")):
            trim = ops.xcorr_planar(srp, tmpl, mma_mode=mode)
            close = float((trim.float() - ref.float()).abs().max() / ref.float().abs().max().clamp_min(1e-6))
            t = time_launches(lambda: check(L.smot_xcorr_planar_mode(ops._ptr(srp), ops._ptr(tmpl), ops._ptr(got), n, Cc, mode,
                                                                     stream_ptr()), "xcorr_planar"))
            t["max_rel_diff_vs_default"] = round(close, 6)
            res["xcorr_planar"][key] = t
    except Exception as exc:
        res["xcorr_planar"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    return res


# --------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes oracle/)
# --------------------------------------------------------------------------------------------------
def oracle_runner():
    from oracle.siammot_oracle import OracleSiamMOT, build_memory
    from siammot_b200.synthetic import make_state_dict
    from oracle import preprocess as opp
    cfg = build_cfg("float32")
    orc = OracleSiamMOT(cfg, make_state_dict(cfg, 1))
    frames = [opp.preprocess(f.numpy(), cfg) for f in make_frames_u8(4, cfg)]   # same frames, test transform on the CPU
    boxes = track_table()
    feats = orc.features(frames[0])
    orc.pool.reset()
    ids = torch.tensor([orc.pool.start() for _ in range(N_TRACKS)])
    det = dict(boxes=boxes, scores=torch.full((N_TRACKS,), 0.9), ids=ids, labels=torch.ones(N_TRACKS, dtype=torch.int64))
    mem = build_memory(orc.P, cfg, orc.pool, feats, det)
    orc.pool.frame += 1
    snap = (set(orc.pool.active), dict(orc.pool.dormant), dict(orc.pool.cache), orc.pool.next_id, orc.pool.frame)

    def step(i):
        orc.pool.active, orc.pool.dormant, orc.pool.cache = set(snap[0]), dict(snap[1]), dict(snap[2])
        orc.pool.next_id, orc.pool.frame = snap[3], snap[4]
        orc.memory = mem
        return orc.forward(frames[i % len(frames)])
    return step


def cpu_baseline(sample_frames=2):
    torch.set_num_threads(host_threads())
    step = oracle_runner()
    step(0)
    t0 = time.perf_counter()
    for i in range(sample_frames):
        step(i + 1)
    dt = time.perf_counter() - t0
    return {"value": round(sample_frames / dt, 4), "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d frames of the same workload (704x1280, 30 tracks) through oracle/siammot_oracle.py, fp32, "
                      "after 1 warm-up frame" % sample_frames}


def run_reference(args):
    """--impl reference: the reference algorithm on the host CPU (oracle port), rank 0 only, on every host thread the process
    may use (torchrun exports OMP_NUM_THREADS=1: overridden here), same workload / config keys / warm-up count as our arm."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = host_threads()
    torch.set_num_threads(cores)
    step = oracle_runner()
    warm = max(args.warmup, 0)
    for i in range(warm):
        step(i)
    steps = args.steps
    ntrk = 0
    t0 = time.perf_counter()
    for i in range(steps):
        out = step(warm + i)
        ntrk += int((out["ids"] >= 0).sum())
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out["boxes"], out["scores"], out["ids"], out["labels"])
    fps = steps / dt
    world = int(os.environ.get("WORLD_SIZE", 1)) if (args.gpus > 1 and "RANK" in os.environ) else 1
    cfgd = config_dict(world)
    cfgd["tracked_boxes_per_step"] = round(ntrk / steps, 1)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(fps, 4), "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": round(dt / steps * 1e3, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfgd,
        "notes": {"what": "reference algorithm on the host CPU (oracle port, fp32; the reference itself needs maskrcnn_benchmark which "
                          "is not installable offline); rank 0 only, %d torch threads" % cores},
        "cpu_baseline": {"value": round(fps, 4), "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "%d full frames (%dx%d, %d tracks) after %d warm-up frames" % (steps, H_NET, W_NET, N_TRACKS, warm)},
        "e2e": {"value": round(fps, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="float16", choices=["float16", "float32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--experimental", default="off", choices=["subprocess", "inproc", "off", "child"],
                    help="information-only A/B arms of the pipeline switches (all of them are measured defaults since round 2, so "
                         "this is off unless asked for): in a child process after the line is final, in this process under a "
                         "watchdog (tests), or not at all (default); 'child' is the child's mode")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's result (boxes, scores, ids, labels) as DIR/<name>.npy")
    ap.add_argument("--workload", default="720p30", choices=sorted(WORKLOADS),
                    help="720p30 = BASELINE.json configs[1] (the metric's configuration, default); 1080p80 = configs[2]; "
                         "r50_720p30 = configs[4]")
    args = ap.parse_args()
    select_workload(args.workload)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.experimental == "child":
        run_experimental_child(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
