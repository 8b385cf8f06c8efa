#!/usr/bin/env python
"""bench.py -- headline benchmark of the dense optical-flow hot path (BASELINE.json metric:
1080p frame-pairs/s, TV-L1 and Farneback, at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload tvl1|farneback|tvl1_4k]
                    [--dump-outputs DIR]

One rank per GPU (torchrun for N > 1).  A *step* is one pass of the hot path over one batch of synthetic frame
pairs (`--pairs` per GPU, default 32: 133 MB of u8 input per step at 1080p, larger than the 126 MB L2).  Frame
pairs are independent, so ranks share nothing on the data path (weak scaling); with N > 1 every step ends with
the NCCL gather of every flow field to rank 0, inside the timed region.

The printed JSON line (rank 0) is the record of the HEADLINE workload (BASELINE configs[2]: TV-L1 1080p, 5 scales /
10 warps / 30 iterations, epsilon = 0) with the base contract's keys plus
  roofline      dominant kernel class: SURVEY §8d algorithmic bytes / CUDA-event launch time / measured HBM peak (`frac`),
                next to what the hardware really did: `dram_frac` (ncu dram bytes / duration / peak), `issue_active`,
                `valid_fraction` (share of computed pixels that are not halo).  Measured on ONE stream (`streams: 1`,
                every launch bracketed by CUDA events on the launching stream); `value_1stream` is the pairs/s of that
                same single-stream mode so the two can be reconciled with the batched `value`;
  cpu_baseline  the reference's CPU path on the host cores (bounded sample);
  e2e           same metric through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region),
                over the same 32-pair batches for >= 2 s;
and two sub-records measured the same way in the same run, so BENCH/SCALE cover the whole BASELINE metric:
  farneback     BASELINE configs[1] (cv::cuda::FarnebackOpticalFlow 1080p, 5 levels) -- value, e2e, roofline, cpu_baseline
  tvl1_4k       BASELINE configs[4] (batched TV-L1 on 3840x2160 pairs, 32 pairs per GPU, NCCL gather) -- value, e2e
`--workload X` makes X the top-level record instead (and skips the sub-records).
`--dump-outputs DIR` writes the flows of each workload's last timed step to DIR/<workload>_flow.npy (see dump_flows);
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import glob
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# NCCL's INFO log goes to a file per process (stdout must stay one JSON line); rank 0 copies the communicator
# lines ("... nranks N ...") to stderr and into the JSON line after the run, so the rank count stays checkable.
NCCL_LOG_DIR = None
if int(os.environ.get("WORLD_SIZE", "1")) > 1:
    NCCL_LOG_DIR = tempfile.mkdtemp(prefix="b200flow-nccl-")  # outside the tree, which may be read-only
    os.environ.setdefault("NCCL_DEBUG", "INFO")
    if os.environ["NCCL_DEBUG"].upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "INFO"
    os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(NCCL_LOG_DIR, "nccl.%h.%p.log"))
else:
    os.environ.pop("NCCL_DEBUG", None)  # some boxes export NCCL_DEBUG=VERSION, which prints a banner to stdout

WORKLOADS = {
    # BASELINE.json configs[2] / north_star target: TV-L1 1080p, 5 scales / 10 warps / 30 iters, epsilon = 0
    # (fixed work, SURVEY.md §8d)
    "tvl1": dict(name="cv::cuda::OpticalFlowDual_TVL1 1920x1080 u8, 5 scales/10 warps/30 iters, epsilon=0",
                 family="tvl1", H=1080, W=1920, dtype="f32", unit="1080p frame-pairs/s", streams=4,
                 params=dict(tau=0.25, lambda_=0.15, theta=0.3, nscales=5, warps=10, epsilon=0.0, iterations=30,
                             scale_step=0.8, gamma=0.0, use_initial_flow=0)),
    # BASELINE.json configs[1]: Farneback 1080p, 5 pyramid levels (perf_optflow.cpp:242-258)
    "farneback": dict(name="cv::cuda::FarnebackOpticalFlow 1920x1080 u8, numLevels=5 pyrScale=0.5 winSize=13 "
                           "numIters=10 polyN=5 polySigma=1.1", family="farneback", H=1080, W=1920, dtype="f32",
                      unit="1080p frame-pairs/s", streams=8,
                      params=dict(num_levels=5, pyr_scale=0.5, fast_pyramids=0, win_size=13, num_iters=10, poly_n=5,
                                  poly_sigma=1.1, flags=0)),
    # BASELINE.json configs[4]: batched TV-L1 on 3840x2160 pairs, 32 per GPU (256 over 8 GPUs), NCCL gather
    "tvl1_4k": dict(name="batched cv::cuda::OpticalFlowDual_TVL1 3840x2160 u8, 5 scales/10 warps/30 iters, epsilon=0, "
                         "32 pairs per GPU", family="tvl1", H=2160, W=3840, dtype="f32", unit="4K frame-pairs/s",
                    streams=4,
                    params=dict(tau=0.25, lambda_=0.15, theta=0.3, nscales=5, warps=10, epsilon=0.0, iterations=30,
                                scale_step=0.8, gamma=0.0, use_initial_flow=0)),
}


def make_alg(workload: str):
    import opencv_contrib_b200 as ocb
    if WORKLOADS[workload]["family"] == "tvl1":
        return ocb.OpticalFlowDual_TVL1_create(tau=0.25, lambda_=0.15, theta=0.3, nscales=5, warps=10, epsilon=0.0,
                                               iterations=30, scaleStep=0.8, gamma=0.0, useInitialFlow=False)
    return ocb.FarnebackOpticalFlow_create(numLevels=5, pyrScale=0.5, fastPyramids=False, winSize=13, numIters=10,
                                           polyN=5, polySigma=1.1, flags=0)


def texture(h: int, w: int, seed: int, cell: int = 8, sigma: float = 1.5):
    """Low-pass random texture in [0, 255] float32 (two octaves of uniform noise, bicubic upsampling, Gaussian
    blur, contrast stretch) -- input synthesis only, outside every timed region."""
    import numpy as np
    import cv2
    rng = np.random.default_rng(seed)
    gh, gw = (h + cell - 1) // cell + 2, (w + cell - 1) // cell + 2
    coarse = rng.random((gh, gw), dtype=np.float32)
    coarse2 = rng.random(((gh + 3) // 4 + 2, (gw + 3) // 4 + 2), dtype=np.float32)
    up = cv2.resize(coarse, (gw * cell, gh * cell), interpolation=cv2.INTER_CUBIC)
    up2 = cv2.resize(coarse2, (gw * cell, gh * cell), interpolation=cv2.INTER_CUBIC)
    img = cv2.GaussianBlur((up + 1.5 * up2)[cell:cell + h, cell:cell + w], (0, 0), sigma)
    lo, hi = float(img.min()), float(img.max())
    return ((img - lo) * (255.0 / max(hi - lo, 1e-6))).astype(np.float32)


def synth_frames(n_frames: int, H: int, W: int, seed: int = 0):
    """n_frames distinct u8 frames; pair i = (frame i, frame i+1) of a drifting texture (3 px right per frame plus a
    vertical sway of +-8 px)."""
    import numpy as np
    T = texture(H + 64, W + 64 + 3 * n_frames, seed)
    frames = []
    for i in range(n_frames):
        dy = int(round(8 * np.sin(i * 0.7)))
        frames.append(np.clip(np.rint(T[32 + dy:32 + dy + H, 3 * i:3 * i + W]), 0, 255).astype(np.uint8))
    return frames


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def sample_now(self):
        """One synchronous query (used while work is still queued on the GPU, so short timed regions -- a few
        Farneback steps finish faster than the 200 ms polling period -- still get a sample under load)."""
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            self.lines.extend(l.strip() for l in out.splitlines() if l.strip())
        except Exception:
            pass

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
                power.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def peak_hbm_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ CPU arms
def cpu_reference_run(workload: str, steps: int, warmup: int, budget_s: float = 25.0):
    """Times the reference's CPU implementation of the path on the host cores, on a bounded sample of the
    workload (whole 1080p pairs until `steps` or `budget_s` is reached; the value is pairs / total seconds).
    Farneback: the LIVE reference cv2.calcOpticalFlowFarneback (kind 'reference').
    TV-L1: oracle/_ref/libtvl1_ref.so = the reference's own modules/optflow/src/tvl1flow.cpp compiled unmodified
    (kind 'reference'; its three imgproc primitives are the cv2-pinned restatements), else the bit-identical
    C/OpenMP port (kind 'port'), else the numpy restatement on a crop."""
    import cv2
    spec = WORKLOADS[workload]
    H, W = spec["H"], spec["W"]
    frames = synth_frames(2, H, W)
    I0, I1 = frames[0], frames[1]
    cores = os.cpu_count() or 1
    scale = 1.0
    if spec["family"] == "farneback":
        cv2.setNumThreads(-1)

        def one():
            cv2.calcOpticalFlowFarneback(I0, I1, None, 0.5, 5, 13, 10, 5, 1.1, 0)

        used = cv2.getNumThreads()
        kind, sample = "reference", "whole %dx%d pairs, cv2 %s calcOpticalFlowFarneback, %d threads" % (
            W, H, cv2.__version__, used)
    else:
        from oracle import tvl1_cpu, tvl1_cpu_native, tvl1_ref
        P = tvl1_cpu.TVL1Params(tau=0.25, lambda_=0.15, theta=0.3, nscales=5, warps=10, epsilon=0.0,
                                innerIterations=1, outerIterations=30, scaleStep=0.8, gamma=0.0, medianFiltering=1)
        n_thr = tvl1_cpu_native.usable_cpus()
        if tvl1_ref.available():
            used = tvl1_ref.set_threads(n_thr)

            def one():
                tvl1_ref.calc(I0, I1, P)
            kind = "reference"
            sample = ("whole %dx%d pairs, the reference's optflow/src/tvl1flow.cpp compiled unmodified (oracle/_ref), "
                      "OpenMP parallel_for_, %d threads (host reports %d logical CPUs)" % (W, H, used, cores))
        elif tvl1_cpu_native.available():
            used = tvl1_cpu_native.set_threads(n_thr)

            def one():
                tvl1_cpu_native.calc(I0, I1, P)
            kind = "port"
            sample = ("whole %dx%d pairs, C/OpenMP port of optflow/src/tvl1flow.cpp, %d threads (host reports %d "
                      "logical CPUs)" % (W, H, used, cores))
        else:
            c0, c1 = I0[:270, :480].copy(), I1[:270, :480].copy()

            def one():
                tvl1_cpu.calc(c0, c1, P)
            kind, scale, used = "port", (270 * 480) / float(H * W), 1
            sample = "480x270 crop per step, numpy restatement, value scaled by area"
    for _ in range(max(0, min(warmup, 1))):
        one()
    times = []
    t_all = time.perf_counter()
    while len(times) < steps:
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    dt = sum(times)
    times.sort()
    return dict(value=len(times) * scale / dt, unit=spec["unit"], cores=used, kind=kind, sample=sample,
                steps_run=len(times), seconds=dt, best=scale / times[0], median=scale / times[len(times) // 2])


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    wl = args.workload or "tvl1"
    r = cpu_reference_run(wl, args.steps, args.warmup, budget_s=120.0)
    spec = WORKLOADS[wl]
    line = {
        "impl": "reference", "metric": "1080p frame-pairs/sec (%s)" % wl, "value": r["value"],
        "unit": spec["unit"], "n_gpus": args.gpus, "steps": r["steps_run"], "warmup": min(args.warmup, 1),
        "ms_per_step": 1000.0 * r["seconds"] / max(r["steps_run"], 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": spec["dtype"], "data": "synthetic",
        "config": {"workload": spec["name"], "pairs_per_step": 1},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "best", "median")},
        "e2e": {"value": r["value"], "unit": spec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def side_measurements(pairs, flow_views, dev, H, W):
    """Secondary single-stream numbers for the other BASELINE configs (not the headline `value`):
    device-resident, CUDA events, after the main timed region."""
    import torch
    import opencv_contrib_b200 as ocb
    out = {}

    side = torch.cuda.Stream()  # a real stream: the legacy default stream takes the no-graph, device-synchronising path

    def time_alg(alg, a, b, f, n):
        torch.cuda.synchronize()
        for _ in range(2):
            alg.calc(a, b, f, side)
        side.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for _ in range(n):
            alg.calc(a, b, f, side)
        e1.record(side)
        side.synchronize()
        return 1000.0 * n / e0.elapsed_time(e1)

    a, b = pairs[0]
    f = flow_views[0]
    try:
        # the reference's create() defaults (5 warps, <= 300 iterations, epsilon 0.01: data-dependent early exit)
        alg = ocb.OpticalFlowDual_TVL1_create()
        out["tvl1_1080p_reference_defaults_eps0.01_pairs_per_s_1stream"] = time_alg(alg, a, b, f, 5)
        out["tvl1_1080p_reference_defaults_iterations_run"] = alg.getStats()["iterations_run"]
        # BASELINE configs[3]: Brox 1280x720, the reference's only parameter set (10, 77, 10)
        bx = (a[:720, :1280].float() / 255.0).contiguous()
        by = (b[:720, :1280].float() / 255.0).contiguous()
        bf = torch.empty((720, 1280, 2), dtype=torch.float32, device=dev)
        alg = ocb.BroxOpticalFlow_create(0.197, 50.0, 0.8, 10, 77, 10)
        out["brox_720p_10_77_10_pairs_per_s_1stream"] = time_alg(alg, bx, by, bf, 3)
        alg.resetStats()
        alg.calc(bx, by, bf, side)
        side.synchronize()
        out["brox_720p_launches_per_pair"] = alg.getStats()["launches"]
        out["denselk_1080p_default_pairs_per_s_1stream"] = time_alg(ocb.DensePyrLKOpticalFlow_create(), a, b, f, 3)
        # video front end (one upload per frame, 3-stream pipeline): host frames in, host flows out
        import numpy as np
        hf = [x.cpu().numpy() for (x, _) in pairs[:9]]
        for name, make in (("tvl1_5x10x30_eps0", lambda: ocb.OpticalFlowDual_TVL1_create(nscales=5, warps=10, epsilon=0.0,
                                                                                       iterations=30)),
                           ("farneback_default", lambda: ocb.FarnebackOpticalFlow_create())):
            vf = ocb.VideoFlow(make(), H, W, dtype=np.uint8, depth=3)
            seq = [hf[i % len(hf)] for i in range(25)]
            for _ in vf.run(seq[:4], copy=False):
                pass
            t0 = time.perf_counter()
            n = sum(1 for _ in vf.run(seq, copy=False))
            out["video_%s_1080p_pairs_per_s_host_to_host" % name] = n / (time.perf_counter() - t0)
            vf.close()
        # interpolateFrames, the consumer right after calc (cudalegacy), 1080p
        u, v = (torch.randn((H, W), device=dev) * 3 for _ in range(2))
        f0, f1 = a.float() / 255.0, b.float() / 255.0
        mid, buf = torch.empty_like(f0), torch.empty((6 * H, W), device=dev)
        for _ in range(2):
            ocb.interpolateFrames(f0, f1, u, v, -u, -v, 0.5, mid, buf)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            ocb.interpolateFrames(f0, f1, u, v, -u, -v, 0.5, mid, buf)
        e1.record()
        torch.cuda.synchronize()
        out["interpolate_frames_1080p_frames_per_s"] = 20000.0 / e0.elapsed_time(e1)
    except Exception as e:  # side numbers must never break the headline line
        out["error"] = repr(e)
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def ncu_facts(kernel_class: str):
    """What ncu measured for this kernel class (committed capture, profiles/r02_traffic.json; r01 as fallback):
    DRAM bytes and duration of one launch, issue-slot utilisation."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", name))).get(kernel_class)
            if tr:
                tr = dict(tr)
                tr["source"] = "profiles/" + name
                return tr
        except Exception:
            continue
    return None


def single_stream_roofline(workload: str, pairs, flow_views, B: int):
    """Roofline record of the dominant kernel class, measured on ONE stream: every launch bracketed by CUDA events
    on the launching stream (engine profiling mode), plus the pairs/s of the same single-stream mode (CUDA graph
    path, as in production) so that launch times, share and throughput describe one execution mode."""
    import torch
    alg = make_alg(workload)
    side = torch.cuda.Stream()  # a real stream: the legacy default stream takes the no-graph, device-synchronising path
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        alg.calc(*pairs[0], flow_views[0], side)
        side.synchronize()
        # throughput of the single-stream mode
        n1 = min(B, 8)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for i in range(n1):
            alg.calc(*pairs[i], flow_views[i], side)
        e1.record(side)
        side.synchronize()
        value_1 = 1000.0 * n1 / e0.elapsed_time(e1)
        # per-launch events
        alg.setProfiling(True)
        alg.resetStats()
        n_prof = min(3, B)
        for i in range(n_prof):
            alg.calc(*pairs[i], flow_views[i], side)
        side.synchronize()
    torch.cuda.synchronize()
    st = alg.getStats()
    alg.setProfiling(False)
    dom_name, dom = max(st["classes"].items(), key=lambda kv: kv[1]["ms"])
    peak, peak_src = peak_hbm_gbs()
    ach = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9 if dom["ms"] > 0 else 0.0
    total_ms = max(sum(c["ms"] for c in st["classes"].values()), 1e-9)
    r = {"bound": "hbm", "kernel": dom_name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
         "traffic": None, "peak_source": peak_src, "streams": 1, "value_1stream": value_1,
         "ms_per_pair_1stream_profiled": total_ms / n_prof,
         "launches_timed": dom["launches"], "avg_launch_us": 1e3 * dom["ms"] / max(dom["launches"], 1),
         "share_of_step": dom["ms"] / total_ms,
         "algorithmic_bytes_per_launch": dom["bytes"] / max(dom["launches"], 1),
         "how": "single stream; CUDA events around every launch on the launching stream (engine profiling mode, no "
                "CUDA graph); value_1stream = same stream, CUDA-graph path; frac counts SURVEY 8d algorithmic bytes, "
                "so K fused iterations per HBM pass push it above 1 -- dram_frac is the hardware's view",
         "all_classes_ms_per_pair": {k: v["ms"] / n_prof for k, v in st["classes"].items()}}
    if dom_name == "tvl1_iter":
        r["valid_fraction"] = (64 - 16) ** 2 / 64.0 ** 2  # K = 8: 8-pixel halo on a 64x64 region
        r["fused_iterations_per_launch"] = "8+8+8+6"
    facts = ncu_facts(dom_name)
    if facts:
        r["traffic"] = facts.get("dram_bytes_per_launch")
        r["traffic_launch"] = facts.get("launch")
        r["traffic_algorithmic_bytes"] = facts.get("algorithmic_bytes_per_launch")
        if facts.get("duration_us") and facts.get("dram_bytes_per_launch"):
            r["dram_frac"] = facts["dram_bytes_per_launch"] / (facts["duration_us"] * 1e-6) / 1e9 / peak
        for k in ("issue_active", "duration_us", "pipe_fma", "pipe_xu", "source"):
            if facts.get(k) is not None:
                r["ncu_" + k] = facts[k]
    return r


DUMP_SAMPLES = 1 << 21  # flow vectors per workload: 16 MB of float32, 48 MB for the three workloads of a default run


def dump_flows(out_dir: str, name: str, flows):
    """Writes out_dir/<name>.npy, float32: the (pairs, H, W, 2) flows when they hold at most DUMP_SAMPLES vectors,
    else a fixed sample of DUMP_SAMPLES of them, shape (DUMP_SAMPLES, 2): flat (pair, y, x) positions drawn with
    numpy's default_rng(0) and sorted, the same for every run with the same --pairs and workload."""
    import numpy as np
    import torch
    n = flows.numel() // 2
    if n <= DUMP_SAMPLES:
        out = flows.cpu().numpy()
    else:
        idx = np.sort(np.random.default_rng(0).integers(0, n, DUMP_SAMPLES))
        out = flows.reshape(-1, 2)[torch.from_numpy(idx).to(flows.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), out)


def measure(workload: str, args, rank: int, world: int, dev, steps: int, sampler=None):
    """One workload, measured like the contract says: W warm-up steps, then `steps` steps between a barrier +
    synchronize on both sides, CUDA events, max over ranks; then the e2e leg over the same batches."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from opencv_contrib_b200.batch import NativeFlowBatch, gather_flows

    spec = WORKLOADS[workload]
    H, W = spec["H"], spec["W"]
    B = args.pairs
    streams = args.streams if args.streams > 0 else spec["streams"]
    frames_h = synth_frames(B + 1, H, W, seed=rank)
    frames = [torch.from_numpy(f).to(dev) for f in frames_h]
    pairs = [(frames[i], frames[i + 1]) for i in range(B)]
    flows = torch.empty((B, H, W, 2), dtype=torch.float32, device=dev)
    flow_views = [flows[i] for i in range(B)]
    # native batch front end (csrc/batch.cu): N engine handles on N streams, one C call per batch
    batcher = NativeFlowBatch(spec["family"], spec["params"], n_streams=streams)
    comm = NATIVE_COMM.get("comm") if (world > 1 and args.gather == "native") else None
    gathered = None
    if world > 1 and rank == 0:  # native: rank 0's own flows are computed straight into their slot
        gathered = [flows if (r == 0 and comm is not None) else torch.empty_like(flows) for r in range(world)]

    def step():
        if comm is not None:   # per-pair ncclSend / ncclRecv on the library's communication stream, overlapped with the solves
            batcher.run_device_gather(pairs, flow_views, comm, 0, gathered)
        else:
            batcher.run_device(pairs, flow_views)
            if world > 1:      # one torch.distributed.gather after the whole batch
                gather_flows(flows, dst=0, out=gathered)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    batcher.reset_stats()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    if sampler is not None:
        sampler.sample_now()  # the steps above are asynchronous: the GPU is still working through them
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if sampler is not None else None
    if args.dump_outputs and rank == 0:  # before the legs below reuse the flow buffers
        dump_flows(args.dump_outputs, workload + "_flow", flows)
    total_ms = float(ms.item())
    launches = batcher.launches()
    rec = {"value": world * B * steps / (total_ms / 1000.0), "unit": spec["unit"], "steps": steps,
           "warmup": args.warmup, "ms_per_step": total_ms / steps, "gpu_launches": int(launches),
           "config": {"workload": spec["name"], "pairs_per_step_per_gpu": B, "streams_per_gpu": streams,
                      "parallelism": "pairs sharded over %d rank(s)%s" % (
                          world, (", NCCL gather of flows to rank 0 inside the step (%s)" % (
                              "native: per-pair ncclSend/ncclRecv overlapped with the solves" if comm is not None
                              else "torch.distributed.gather after the batch")) if world > 1 else ""),
                      "l2": "inputs per step (%.0f MB u8) exceed the 126 MB L2; engine working set ~%.1f GB/pair" % (
                          B * 2 * H * W / 1e6, 0.3 * H * W / (1080 * 1920))}}
    if clocks is not None:
        rec["clocks"] = clocks
    gathered = None

    # ---- e2e: host (pinned) buffers through b2f_batch_run_host -> b2f_calc_host, copies inside the timed region,
    #      the same B-pair batches, repeated for >= 2 s; every rank runs its shard, the slowest rank sets the time ----
    h_in = [torch.from_numpy(f).pin_memory() for f in frames_h]
    h_out = torch.empty((B, H, W, 2), dtype=torch.float32).pin_memory()
    hp = [(h_in[i].numpy(), h_in[i + 1].numpy()) for i in range(B)]
    ho = [h_out[i].numpy() for i in range(B)]
    batcher.run_host(hp, ho)
    est = rec["ms_per_step"] / 1000.0 * 1.1
    n_e2e = max(2, min(40, int(math.ceil(2.0 / max(est, 1e-3)))))
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        batcher.run_host(hp, ho)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    rec["e2e"] = {"value": world * B * n_e2e / float(dt.item()), "unit": spec["unit"],
                  "h2d_bytes_per_step": world * B * 2 * H * W, "d2h_bytes_per_step": world * B * H * W * 8,
                  "pairs_per_step": world * B, "steps": n_e2e, "seconds": float(dt.item()), "streams": streams,
                  "timing": "host wall clock (max over ranks) around b2f_batch_run_host calls; each returns after the "
                            "last flow's D2H completed"}
    del h_out, h_in
    return rec, pairs, flow_views


NATIVE_COMM = {}


def nccl_init_lines(world: int):
    """Communicator lines of this run's NCCL INFO logs (rank 0's view of `nranks`)."""
    out = []
    for p in sorted(glob.glob(os.path.join(NCCL_LOG_DIR, "nccl.*.%d.log" % os.getpid()))):
        try:
            for ln in open(p, errors="replace"):
                if "nranks" in ln and ("Init COMPLETE" in ln or "comm 0x" in ln):
                    out.append(ln.strip())
        except Exception:
            pass
    return out[:4]


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        if args.gather == "native":
            # the gather is not part of the compute path: if the library cannot create its communicator on this box
            # (no libnccl.so.2 to dlopen, id exchange failed) the run goes on with torch.distributed.gather and says so
            from opencv_contrib_b200.batch import NativeComm
            ok = torch.ones(1, device=dev)
            try:
                NATIVE_COMM["comm"] = NativeComm.from_torch_distributed()
            except Exception as e:  # noqa: BLE001
                NATIVE_COMM["error"] = repr(e)
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # all ranks take the same path
            if float(ok.item()) == 0.0:
                NATIVE_COMM.pop("comm", None)
                if rank == 0:
                    print("native NCCL gather unavailable (%s): using torch.distributed.gather" % NATIVE_COMM.get("error", "another rank failed"),
                          file=sys.stderr, flush=True)

    head = args.workload or "tvl1"
    sampler = ClockSampler(local_rank) if rank == 0 else None
    rec, pairs, flow_views = measure(head, args, rank, world, dev, args.steps, sampler)
    spec = WORKLOADS[head]
    line = None
    if rank == 0:
        line = {"metric": "1080p frame-pairs/sec (%s)" % head if spec["H"] == 1080 else "4K frame-pairs/sec (%s)" % head,
                "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": spec["dtype"], "data": "synthetic", "config": rec["config"],
                "roofline": single_stream_roofline(head, pairs, flow_views, args.pairs),
                "cpu_baseline": None, "e2e": rec["e2e"], "gpu_launches": rec["gpu_launches"],
                "clocks": rec.get("clocks")}
        if not args.no_cpu:
            r = cpu_reference_run(head, steps=5, warmup=1, budget_s=25.0)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "best", "median")}
        if not args.no_extras and spec["H"] == 1080:
            line["extras"] = side_measurements(pairs, flow_views, dev, spec["H"], spec["W"])
    del pairs, flow_views
    torch.cuda.empty_cache()

    if args.workload is None:  # default run: the rest of BASELINE.metric as sub-records, every rank takes part
        for sub in ("farneback", "tvl1_4k"):
            try:
                r2, p2, f2 = measure(sub, args, rank, world, dev, args.steps, None)
                if rank == 0:
                    if sub == "farneback":
                        r2["roofline"] = single_stream_roofline(sub, p2, f2, args.pairs)
                        if not args.no_cpu:
                            c = cpu_reference_run(sub, steps=8, warmup=1, budget_s=12.0)
                            r2["cpu_baseline"] = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample", "best",
                                                                    "median")}
                    else:
                        r2["pixels_per_pair_vs_1080p"] = 4.0
                        r2["equiv_1080p_pairs_per_s"] = 4.0 * r2["value"]
                    r2["metric"] = "%s frame-pairs/sec (%s)" % ("1080p" if WORKLOADS[sub]["H"] == 1080 else "4K", sub)
                    r2["n_gpus"] = world
                    line[sub] = r2
                del p2, f2
                torch.cuda.empty_cache()
            except Exception as e:  # a sub-record must never lose the headline
                if rank == 0:
                    line[sub] = {"error": repr(e)}
    if rank == 0:
        if world > 1:
            lines = nccl_init_lines(world)
            line["nccl"] = {"world_size": world, "debug_file_dir": NCCL_LOG_DIR, "init_lines": lines}
            for ln in lines:
                print(ln, file=sys.stderr, flush=True)
        print(json.dumps(line), flush=True)
    NATIVE_COMM.clear()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="measure only this workload as the top-level record (default: tvl1 headline + farneback + "
                         "tvl1_4k sub-records)")
    ap.add_argument("--pairs", type=int, default=32, help="frame pairs per step per GPU")
    ap.add_argument("--streams", type=int, default=0,
                    help="engine instances / CUDA streams per GPU (0 = per workload: 4 for tvl1, whose persistent kernels "
                         "fill the GPU on their own; 8 for farneback, whose coarse levels are launch-bound)")
    ap.add_argument("--gather", default="native", choices=["native", "torch"],
                    help="N > 1: result gather through libb200flow's own NCCL communicator (per pair, overlapped) or one "
                         "torch.distributed.gather per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary single-stream measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write each workload's flows of the last timed step (rank 0) to DIR/<workload>_flow.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
