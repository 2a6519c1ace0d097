#!/usr/bin/env python
"""Benchmark of the hot path MarkerDetector::detect on B200 (contract: see README / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C1|C2|C3|C4|C5|C4s4] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload = BASELINE.json configs[3] ("C4"): synthetic 3840x2160 grey frames, 100 Fiducidal markers each,
batch of 256 frames per GPU, the reference's defaults (ADPT_THRES 7/7, LINES refinement, per-marker PnP).  One
"step" = one pass of the whole hot path over one batch.  Frames are independent, so N GPUs = N shards, no collective
on the data path (weak scaling: the same batch size per GPU).  The other BASELINE configs (C1 single reference frame,
C2 1280x720 board with erosion + BoardDetector pose, C3 1080p x 64 SUBPIX, C5 HRM 4K, plus the sigma-4 contour storm
"C4s4") are timed the same way with --config, and briefly inside the default run (key `other_configs`, 1 GPU only).

  value   whole-job frames/s with the batch already resident in HBM (device-timed, max over ranks); ONE context, two
          batches in flight inside the library (ab_enqueue_batch_device twice before ab_fetch_results)
  e2e     the same through the C ABI call ab_detect_batch with HOST (pinned) frames: H2D + kernels + D2H
  roofline  the dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured HBM peak
  cpu_baseline  the CPU oracle port (oracle/aruco_oracle.cpp) on a bounded sample: frame-parallel on all host threads
          (value), in the reference's own threading model (ar_omp.h: one frame at a time, OpenMP only at
          markerdetector.cpp:456/587) and the cv2-backed oracle

--impl reference times that CPU oracle port with all host threads on the FIRST frames of the same batch (the
reference's own C++ cannot be built here: no OpenCV C++ -- DESIGN.md section 3).

--dump-outputs DIR writes, after the timed steps, the markers the last timed step returned for the batch (rank 0's shard) as
DIR/<name>.npy, float32/float64: frames (frame index), counts (markers per frame), ids, corners [n,4,2], rvec and tvec [n,3]
(NaN where a marker has no pose), flattened over the markers in frame order.  The frames are generated from fixed seeds, so
two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

MARKER_SIZE = 0.05
N_BASE = 8  # distinct rendered scenes; every frame of a batch gets its own noise realisation
# kernels launched per batch: threshold, scan_starts, trace, trace_long, emit, polygon, frame_filter,
# homography, sample, otsu, identify, refine, finalize, pose (+ erode when erosion is on)
KERNELS_PER_BATCH = 14

CONFIGS = {
    "C1": dict(workload="C1: reference frame testdata/single 640x480 (tests/golden), Fiducidal, ADPT_THRES 7/7 + LINES + PnP, one frame per call",
               W=640, H=480, batch=1, golden="single", size=1.0, params={}),
    "C2": dict(workload="C2: synthetic 1280x720 board frame, 24 Fiducidal markers, erosion on, LINES + BoardDetector pose, one frame per call",
               W=1280, H=720, batch=1, n=24, marker_px=100, sigma=1.5, board=True, params=dict(erosion=True)),
    "C3": dict(workload="C3: synthetic 1920x1080 grey, 50 Fiducidal markers/frame, ADPT_THRES 7/7 + SUBPIX + PnP",
               W=1920, H=1080, batch=64, n=50, sigma=2.0, params=dict(corner_method=2)),
    "C4": dict(workload="C4: synthetic 3840x2160 grey, 100 Fiducidal markers/frame, ADPT_THRES 7/7 + LINES + PnP",
               W=3840, H=2160, batch=256, n=100, sigma=2.0, params={}),
    "C5": dict(workload="C5: synthetic 3840x2160 grey, 100 HRM d6x6 markers/frame, ADPT_THRES 21/7, erosion on, LINES + PnP, warp 64, minSize 0.005",
               W=3840, H=2160, batch=64, n=100, sigma=2.0, hrm="d6x6_100", max_cands=1024,
               params=dict(p1=21, p2=7, warp_size=64, min_size=0.005, decoder=1, erosion=True)),
    "C4s4": dict(workload="C4s4: C4 at noise sigma 4 (contour storm: ~10x the border pixels of sigma 2)",
                 W=3840, H=2160, batch=64, n=100, sigma=4.0, params={}),
    # the round-1 generator (175 px markers: ~5 % of them fall below the detector's minimum contour length and are rejected,
    # 33 % fewer kept contour points) -- kept so that round-1 and round-2 numbers can be compared on the same frames
    "C4r1": dict(workload="C4r1: C4 with the round-1 marker size (175 px, 94.8 detectable markers/frame)",
                 W=3840, H=2160, batch=256, n=100, sigma=2.0, marker_px=175, params={}),
}
METRIC = {"C4": "frames_per_s_4k_100markers"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner to stdout) must not be
# able to add to it: fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(cfg_name, kernel):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this build
    (profiles/ncu_traffic.json, written from the capture by tools/ncu_traffic.py); None when there is none."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        e = d.get(cfg_name, {}).get(kernel)
        return (float(e["dram_bytes_per_launch"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, dev):
        self.rows, self.proc, self.dev = [], None, dev

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.3)  # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def host_threads():
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1, so do not ask OpenMP)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def bind_to_gpu_numa(local):
    """Pins this rank's threads to the CPUs next to its GPU (NVML's ideal CPU set = the GPU's NUMA node / PCIe root) BEFORE
    any pinned host memory is allocated, so the staging pages are first-touched on that node."""
    info = {"cpus_before": host_threads()}
    global _ALL_CPUS
    _ALL_CPUS = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        try:
            info["numa_node"] = int(pynvml.nvmlDeviceGetNumaNodeId(h))
        except Exception:
            info["numa_node"] = None
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
        info["cpus_bound"] = len(os.sched_getaffinity(0))
        try:
            pci = pynvml.nvmlDeviceGetPciInfo(h)
            info["pci_bus_id"] = pci.busId if isinstance(pci.busId, str) else pci.busId.decode()
        except Exception:
            pass
    except Exception as e:  # NVML missing: leave the affinity alone
        info["note"] = "not bound: %s" % type(e).__name__
    return info


_ALL_CPUS = None


def unbind_cpus():
    """Back to every core the process was given (the CPU baseline legs use all of them)."""
    if _ALL_CPUS:
        try:
            os.sched_setaffinity(0, _ALL_CPUS)
        except Exception:
            pass


def oracle_params(cfg):
    from oracle.cv2_oracle import Params
    return Params(**cfg["params"])


def golden(name):
    fr = np.load(os.path.join(ROOT, "tests", "golden", "frames.npz"))
    exp = json.load(open(os.path.join(ROOT, "tests", "golden", "expected.json")))
    return fr, exp


def hrm_codes(cfg):
    _, exp = golden(None)
    text = exp["dictionaries"][cfg["hrm"]]
    n = int(cfg["hrm"][1])
    return text, [l.split('"')[1] for l in text.splitlines() if l.startswith("marker_")], n


def camera(cfg):
    from aruco_b200 import synth
    if cfg.get("golden"):
        _, exp = golden(None)
        intr = exp["intrinsics"][cfg["golden"]]
        return np.array(intr["K"], np.float32).reshape(3, 3), np.array(intr["D"], np.float32).reshape(-1)[:5]
    return synth.camera_for(cfg["W"], cfg["H"])


def base_scenes(cfg, n_base, rank):
    """Noise-free f32 renderings (CPU, numpy, seeded): scene i of rank r has seed 1000 r + i."""
    from aruco_b200 import synth
    t = time.time()
    kw = {}
    if cfg.get("hrm"):
        _, codes, n = hrm_codes(cfg)
        kw = dict(hrm_codes=codes, hrm_n=n)
    scenes, truths = [], []
    for i in range(n_base):
        img, tr = synth.render_frame(cfg["W"], cfg["H"], cfg["n"], seed=1000 * rank + i, as_float=True, marker_px=cfg.get("marker_px"), **kw)
        scenes.append(img)
        truths.append(tr)
    log("[bench] rendered %d base scenes %dx%d in %.1fs" % (n_base, cfg["W"], cfg["H"], time.time() - t))
    return scenes, truths


def make_frames(cfg, n_frames, rank, dev):
    """[n_frames, H, W] u8 on `dev` (a torch device): scene (i mod n_base) + per-frame Gaussian noise from a torch generator
    seeded 1234 + rank ON THAT DEVICE -- both arms of the benchmark call this, so on the same box they see the same frames."""
    import torch
    W, H = cfg["W"], cfg["H"]
    if cfg.get("golden"):
        fr, _ = golden(None)
        g = torch.from_numpy(np.ascontiguousarray(fr[cfg["golden"]])).to(dev)
        return g[None].repeat(n_frames, 1, 1).contiguous(), None
    n_base = min(N_BASE, max(1, n_frames))
    scenes, truths = base_scenes(cfg, n_base, rank)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    frames = torch.empty((n_frames, H, W), dtype=torch.uint8, device=dev)
    clean = [torch.from_numpy(s).to(dev) for s in scenes]
    for i in range(n_frames):
        noise = torch.randn((H, W), generator=gen, device=dev, dtype=torch.float32) * cfg["sigma"]
        frames[i] = torch.clamp(torch.round(clean[i % n_base] + noise), 0, 255).to(torch.uint8)
    return frames, truths


def board_config(cfg, truth):
    """BoardConfiguration in pixels (board.h:56-97) of a synthetic scene: marker corners on the canvas, centred, y up."""
    cc = np.asarray(truth["canvas_corners"], np.float64)
    cx, cy = cfg["W"] / 2.0, cfg["H"] / 2.0
    markers = []
    for mid, c in zip(truth["ids"], cc):
        markers.append({"id": int(mid), "corners": [[float(x - cx), float(-(y - cy)), 0.0] for x, y in c]})
    return {"mInfoType": 0, "markers": markers}


def config_dict(cfg, B, extra=None):
    d = {"workload": cfg["workload"], "frames_per_gpu_per_step": B, "noise_sigma": cfg.get("sigma"),
         "distinct_scenes": 1 if cfg.get("golden") else min(N_BASE, B), "frame_seed": "torch.Generator(1234 + rank) on the GPU, scenes numpy seed 1000 rank + i",
         "l2": "inputs larger than L2 (batch = %.2f GB per GPU vs 126 MB L2)" % (B * cfg["W"] * cfg["H"] / 1e9) if B * cfg["W"] * cfg["H"] > 126e6
         else "L2 flushed between timed steps (256 MB scratch write)",
         "parallelism": "frame shards, one per GPU, no collective"}
    if extra:
        d.update(extra)
    return d


# ------------------------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------------------------
def cpu_detect_batch(cfg, frames_np, K, D, threads, hrm=None, board=None):
    from oracle import native
    P = oracle_params(cfg)
    res = native.detect_batch(frames_np, P, K, D, cfg.get("size", MARKER_SIZE), hrm=hrm, cap=512 if cfg.get("hrm") else 256, threads=threads)
    if board is not None:  # BoardDetector::detect on the host with real OpenCV (the port has no board stage)
        from oracle import cv2_oracle as o
        for ms in res:
            o.board_detect(ms, board, K, D, cfg.get("size", MARKER_SIZE))
    return res


def run_reference(args):
    """CPU arm: the oracle port, OpenMP frame-parallel over all host threads, on the first frames of the SAME batch the
    GPU arm builds (same scenes, same torch generator; generated on the GPU when there is one)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    from oracle import native
    native.load()
    cfg = CONFIGS[args.config]
    B = args.batch or cfg["batch"]
    threads = host_threads()
    px = cfg["W"] * cfg["H"]
    sample = int(min(B, max(1, min(max(2 * threads, 32), 2.7e8 // px))))  # frames per step: a few CPU-seconds on every thread
    on_gpu = torch.cuda.is_available()
    frames_t, truths = make_frames(cfg, sample, 0, torch.device("cuda", 0) if on_gpu else torch.device("cpu"))
    frames = frames_t.cpu().numpy()
    del frames_t
    K, D = camera(cfg)
    hrm = native.dict_from_yaml_text(hrm_codes(cfg)[0]) if cfg.get("hrm") else None
    board = board_config(cfg, truths[0]) if cfg.get("board") else None
    for _ in range(args.warmup):
        cpu_detect_batch(cfg, frames[:threads], K, D, threads, hrm, board)
    t0 = time.perf_counter()
    nm = 0
    for _ in range(args.steps):
        res = cpu_detect_batch(cfg, frames, K, D, threads, hrm, board)
        nm += sum(len(r) for r in res)
    dt = time.perf_counter() - t0
    fps = args.steps * sample / dt
    line = {"impl": "reference", "metric": METRIC.get(args.config, "frames_per_s_" + args.config), "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "mpix_per_s": fps * px / 1e6,
            "config": config_dict(cfg, B),  # the same dict as the GPU arm's: same workload, same frame generator and seeds
            "reference_sample": "first %d frames of the batch per step (%s)" % (sample, "generated on the GPU: identical to the GPU arm's" if on_gpu else "no GPU: CPU generator, other noise realisations"),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": "%d frames/step x %d steps, oracle/aruco_oracle.cpp OpenMP frame-parallel (reference C++ "
                                       "unbuildable: no OpenCV C++)" % (sample, args.steps)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "markers_per_frame": nm / (args.steps * sample), "gpu_launches": 0}
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class Workload:
    """One config on one GPU: frames resident in HBM, a configured detector (ONE context), the timed loops."""

    def __init__(self, name, B, rank, local, torch):
        from aruco_b200 import FiducidalMarkers, HighlyReliableMarkers, MarkerDetector
        self.torch, self.name, self.cfg, self.B, self.local = torch, name, CONFIGS[name], B, local
        cfg = self.cfg
        self.W, self.H = cfg["W"], cfg["H"]
        self.dev = torch.device("cuda", local)
        self.frames, self.truths = make_frames(cfg, B, rank, self.dev)
        self.K, self.D = camera(cfg)
        self.size = cfg.get("size", MARKER_SIZE)
        self.cap = 512 if cfg.get("hrm") else 128
        self.stream = torch.cuda.Stream(device=self.dev)  # the library runs on an explicit stream of the caller
        det = MarkerDetector(local)
        det.set_stream(self.stream.cuda_stream)
        P = oracle_params(cfg)
        det.setThresholdMethod(P.thres_method)
        det.setThresholdParams(P.p1, P.p2)
        det.setCornerRefinementMethod(P.corner_method)
        det.setMinMaxSize(P.min_size, P.max_size)
        det.setWarpSize(P.warp_size)
        det.enableErosion(P.erosion)
        self.hrm_text = None
        if cfg.get("hrm"):
            self.hrm_text = hrm_codes(cfg)[0]
            HighlyReliableMarkers.loadDictionary(self.hrm_text)
            det.setMakerDetectorFunction(HighlyReliableMarkers.detect)
        else:
            det.setMakerDetectorFunction(FiducidalMarkers.detect)
        det.reserve(self.W, self.H, B, max_candidates=cfg.get("max_cands", 0))
        self.det = det
        self.board = None
        if cfg.get("board"):
            from aruco_b200.board import BoardConfiguration
            self.board_dict = board_config(cfg, self.truths[0])
            self.board = BoardConfiguration.from_dict(self.board_dict)
        self.flush = None
        if B * self.W * self.H <= 126e6:  # inputs fit L2: flush it between timed steps
            self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.stream.synchronize()
        torch.cuda.synchronize()

    # one step, one batch at a time
    def step(self):
        self.det.enqueue_device(self.frames.data_ptr(), self.W, self.H, self.B, self.K, self.D, self.size)
        return self.det.fetch(self.B, self.cap, raw=True)

    def parity(self, n_check):
        """ids exact + corners < 0.01 px + pose < 1e-4 of `n_check` frames spread over the batch against the CPU oracle port."""
        from oracle import native
        buf, counts = self.step()
        P = oracle_params(self.cfg)
        hrm = native.dict_from_yaml_text(self.hrm_text) if self.hrm_text else None
        idx = sorted(set(int(round(i)) for i in np.linspace(0, self.B - 1, min(n_check, self.B))))
        host = self.frames[idx].cpu().numpy()
        refs = native.detect_batch(host, P, self.K, self.D, self.size, hrm=hrm, cap=self.cap, threads=host_threads())
        ok, poses, pose_ok = True, 0, 0
        for f, ref in zip(idx, refs):
            got = [buf[f * self.cap + i] for i in range(counts[f])]
            ok &= [m.id for m in got] == [m["id"] for m in ref]
            if not ok:
                break
            for g, m in zip(got, ref):
                ok &= float(np.abs(np.array(g.corners).reshape(4, 2) - m["corners"]).max()) < 0.01
                if "rvec" in m:
                    poses += 1
                    er = np.abs(np.array(g.rvec) - m["rvec"]).max() / np.abs(m["rvec"]).max()
                    et = np.abs(np.array(g.tvec) - m["tvec"]).max() / np.abs(m["tvec"]).max()
                    pose_ok += bool(er < 1e-4 and et < 1e-4)
        ok &= poses == 0 or pose_ok >= 0.99 * poses
        return {"checked_frames": len(idx), "ids_exact": bool(ok), "corners_within_px": 0.01, "poses_within_1e-4": "%d/%d" % (pose_ok, poses)}, counts

    def run_steps(self, n, flush=False):
        """n steps with two batches in flight inside the ONE context: batch i+1 is enqueued before batch i is fetched.  The
        host side of a step is two C-ABI calls on preallocated buffers (no per-step allocation: a slow host thread would
        show up as idle gaps on the device)."""
        from aruco_b200._lib import ab_marker
        det, lib, total, pending = self.det, self.det._lib, 0, 0
        if getattr(self, "_out", None) is None:
            self._out = (ab_marker * (self.B * self.cap))()
            self._cnt = (C.c_int32 * self.B)()
            self._Kf = np.ascontiguousarray(np.asarray(self.K, np.float32).reshape(9))
            self._Df = np.ascontiguousarray(np.asarray(self.D, np.float32).reshape(-1)[:5])
        Kp, Dp = self._Kf.ctypes.data_as(C.c_void_p), self._Df.ctypes.data_as(C.c_void_p)
        ptr = C.c_void_p(self.frames.data_ptr())
        for _ in range(n):
            if pending == 2:
                det._check(lib.ab_fetch_results(det._h, self._out, self.cap, self._cnt))
                total += sum(self._cnt)
                pending -= 1
            if flush and self.flush is not None:
                with self.torch.cuda.stream(self.stream):
                    self.flush.fill_(1)
            det._check(lib.ab_enqueue_batch_device(det._h, ptr, self.W, self.H, self.W, self.W * self.H, self.B, Kp, Dp, self.size))
            pending += 1
        while pending:
            det._check(lib.ab_fetch_results(det._h, self._out, self.cap, self._cnt))
            total += sum(self._cnt)
            pending -= 1
        return total

    def last_step_outputs(self, budget=64 << 20):
        """What the last step of run_steps() handed its caller (ab_fetch_results: a marker count per frame and that many
        ab_marker records), as float arrays flattened over the markers in frame order.  A batch whose markers could take
        more than `budget` bytes is represented by a fixed, seeded sample of its frames (`frames` lists them)."""
        rec = np.ctypeslib.as_array(self._out).reshape(self.B, self.cap)
        counts = np.ctypeslib.as_array(self._cnt)
        frames = np.arange(self.B)
        per_frame = 16 + 88 * self.cap  # frame index and count; id, corners, rvec, tvec of up to cap markers
        if self.B * per_frame > budget:
            frames = np.sort(np.random.default_rng(0).choice(self.B, budget // per_frame, replace=False))
        m = np.concatenate([rec[f, :counts[f]] for f in frames])
        pose = m["has_pose"][:, None] != 0
        return {"frames": frames.astype(np.float64), "counts": counts[frames].astype(np.float64), "ids": m["id"].astype(np.float64),
                "corners": m["corners"].reshape(-1, 4, 2), "rvec": np.where(pose, m["rvec"], np.nan), "tvec": np.where(pose, m["tvec"], np.nan)}

    def time_resident(self, steps, warmup, barrier, sampler=None):
        torch = self.torch
        self.run_steps(max(warmup, 3))
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        t0 = time.perf_counter()
        n_markers = self.run_steps(steps, flush=True)
        # Device clock: e0 is processed before the first kernel (the library's second slot waits for an event recorded on
        # this stream after e0), e1 is recorded after the last fetch returned, i.e. after every kernel and copy of both
        # in-flight slots has completed.  The host clock over the same region is kept as a cross-check (wall_ms).
        e1.record(self.stream)
        self.stream.synchronize()
        self.wall_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        clocks = sampler.stop() if sampler else None
        ms = e0.elapsed_time(e1)
        if self.flush is not None:  # take the flush writes out again: time them alone
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(self.stream):
                f0.record(self.stream)
                for _ in range(steps):
                    self.flush.fill_(1)
                f1.record(self.stream)
            self.stream.synchronize()
            ms = max(ms - f0.elapsed_time(f1), 1e-3)
        return ms, n_markers, clocks

    def kernel_ms(self, reps=3):
        det = self.det
        det.enable_timing(True)
        self.step()
        acc = {k: 0.0 for k in det.KERNELS}
        for _ in range(reps):
            self.step()
            for k, v in det.kernel_ms().items():
                acc[k] += v / reps
        det.enable_timing(False)
        return acc

    def time_e2e(self, steps, barrier, chunk=32):
        """Through the plugin call with HOST frames: ab_detect_batch (+ ab_detect_board per frame for the board config)."""
        torch = self.torch
        from aruco_b200 import MarkerDetector
        from aruco_b200._lib import ab_marker
        B, W, H, cap = self.B, self.W, self.H, self.cap
        host = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
        host.copy_(self.frames)
        det = self.det
        det.reserve(W, H, min(chunk, B), max_candidates=self.cfg.get("max_cands", 0))  # chunked: H2D of chunk c+1 under the kernels of chunk c
        out = (ab_marker * (B * cap))()
        cnts = (C.c_int32 * B)()
        Kf, Df = np.ascontiguousarray(self.K.reshape(9)), np.ascontiguousarray(self.D)
        board_call = None
        if self.board is not None:
            # BoardDetector::detect (boarddetector.cpp:90-204) through the C ABI on the markers just found: ab_detect_board takes
            # the ab_marker array as ab_detect_batch wrote it (the Python mirror's per-marker marshalling is not timed)
            from aruco_b200._lib import ab_board, ab_board_config
            ids = np.ascontiguousarray(np.array(self.board.ids, np.int32))
            pts = np.ascontiguousarray(self.board.objPoints.astype(np.float32).reshape(-1))
            cfgb = ab_board_config(len(ids), self.board.mInfoType, ids.ctypes.data, pts.ctypes.data)
            outm, resb = (ab_marker * cap)(), ab_board()

            def board_call():
                for f in range(B):
                    frame_markers = (ab_marker * cap).from_buffer(out, f * cap * C.sizeof(ab_marker))
                    det._check(det._lib.ab_detect_board(det._h, frame_markers, cnts[f], C.byref(cfgb), Kf.ctypes.data_as(C.c_void_p),
                                                        Df.ctypes.data_as(C.c_void_p), float(self.size), -1.0, 0, outm, C.byref(resb)))
                    assert resb.has_pose and resb.prob > 0.5

        def one():
            rc = det._lib.ab_detect_batch(det._h, C.c_void_p(host.data_ptr()), W, H, W, W * H, B, Kf.ctypes.data_as(C.c_void_p),
                                          Df.ctypes.data_as(C.c_void_p), self.size, out, cap, cnts)
            det._check(rc)
            if board_call is not None:
                board_call()

        for _ in range(2):
            one()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        self.stream.synchronize()
        ms = (time.perf_counter() - t0) * 1e3  # every call returns after its D2H copy: the host clock is the device clock
        barrier()
        # the host-side ceiling: the same pinned buffer, the same chunking, copies only
        dst = torch.empty((min(chunk, B), H, W), dtype=torch.uint8, device=self.dev)
        cs = torch.cuda.Stream(device=self.dev)
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(cs):
            for rep in range(3):
                if rep == 1:
                    h0.record(cs)
                for c0 in range(0, B, chunk):
                    n = min(chunk, B - c0)
                    dst[:n].copy_(host[c0:c0 + n], non_blocking=True)
            h1.record(cs)
        cs.synchronize()
        h2d_gbs = 2 * B * W * H / (h0.elapsed_time(h1) / 1e3) / 1e9
        det.reserve(W, H, B, max_candidates=self.cfg.get("max_cands", 0))
        same = None
        return ms, {"h2d_bytes_per_step": B * W * H, "d2h_bytes_per_step": B * cap * C.sizeof(ab_marker) + 4 * B,
                    "chunk_frames": min(chunk, B), "h2d_only_gbs": h2d_gbs, "counts": list(cnts)}

    def cpu_baselines(self, budget_px=2.2e9):
        """The oracle port on a bounded sample of this batch: (i) frame-parallel on all host threads, (ii) the reference's own
        threading model (ar_omp.h: one frame at a time, OpenMP inside a frame only at cpp:456/587), (iii) the cv2-backed oracle."""
        from oracle import native
        cfg, threads = self.cfg, host_threads()
        px = self.W * self.H
        sample = int(max(1, min(self.B, budget_px // px)))
        hostf = self.frames[:sample].cpu().numpy()
        hrm = native.dict_from_yaml_text(self.hrm_text) if self.hrm_text else None
        board = self.board_dict if self.board is not None else None
        cpu_detect_batch(cfg, hostf[:min(sample, threads)], self.K, self.D, threads, hrm, board)
        t0 = time.perf_counter()
        cpu_detect_batch(cfg, hostf, self.K, self.D, threads, hrm, board)
        dt = time.perf_counter() - t0
        out = {"value": sample / dt, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": "%d frames of the same batch, oracle/aruco_oracle.cpp, OpenMP frame-parallel on %d threads" % (sample, threads)}
        # (ii) ar_omp model: frames one after the other; orc_detect parallelises only the reference's two omp loops
        n2 = max(1, min(sample, int(4e8 // px)))
        P = oracle_params(cfg)
        t0 = time.perf_counter()
        for f in range(n2):
            native.detect(hostf[f], P, self.K, self.D, self.size, hrm, cap=2048, debug=False)
        out["ar_omp_model"] = {"value": n2 / (time.perf_counter() - t0), "unit": "frames/s", "cores": threads,
                               "sample": "%d frames one at a time; OpenMP only where the reference has it (markerdetector.cpp:456,587)" % n2}
        try:  # (iii) real OpenCV primitives + Python glue, single process (BASELINE.md section 4)
            from oracle import cv2_oracle as o
            hc = o.HrmDictionary.from_yaml_text(self.hrm_text) if self.hrm_text else None
            n3 = max(1, min(sample, int(1e8 // px)))
            t0 = time.perf_counter()
            for f in range(n3):
                o.detect(hostf[f], P, self.K, self.D, self.size, hc)
            out["cv2_oracle"] = {"value": n3 / (time.perf_counter() - t0), "unit": "frames/s", "cores": 1,
                                 "sample": "%d frames, oracle/cv2_oracle.py (OpenCV %s primitives, Python glue)" % (n3, o.cv2.__version__)}
        except Exception as e:
            out["cv2_oracle"] = {"unavailable": type(e).__name__}
        return out


def algorithmic_bytes(kernel, W, H, B, k_thr):
    """Algorithmic bytes per launch (SURVEY.md section 8(d), DESIGN.md section 5): threshold reads the grey frame and writes the
    u8 binarised frame (the 1/8 B/px packed copy is not counted); the scan and the walkers read the packed image; the other
    kernels work per candidate (< 1 % of a frame) and are given the whole-path figure 3 W H."""
    packed = W * H / 8.0 * B
    return {"threshold": 2.0 * W * H * B, "scan_starts": packed, "trace": packed, "trace_long": packed, "emit": packed}.get(kernel, 3.0 * W * H * B)


def measure_config(name, args, rank, local, world, torch, dist, full):
    """Times one config on this rank.  full: the whole protocol (parity gate on >= 16 frames, clocks, e2e, CPU baselines);
    otherwise the short form used for `other_configs`."""
    cfg = CONFIGS[name]
    B = args.batch if (args.batch and full) else cfg["batch"]
    wl = Workload(name, B, rank, local, torch)
    W, H = wl.W, wl.H

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity, counts = ({"checked_frames": 0, "ids_exact": None}, None)
    if rank == 0:
        parity, counts = wl.parity(16 if full else 4)
        log("[bench] %s parity vs oracle: %s; markers/frame=%.1f counters=%s" % (name, parity, float(np.mean(counts)), wl.det.counters()))
        if not parity["ids_exact"]:
            raise SystemExit("parity check against the oracle failed (%s) -- refusing to report a number" % name)
    steps = args.steps if full else max(5, min(args.steps, 20))
    if B == 1 and not full:
        steps = max(steps, 200)  # single-frame configs timed on the side: enough calls for a stable latency
    sampler = ClockSampler(local) if (rank == 0 and full) else None
    ms, n_markers, clocks = wl.time_resident(steps, args.warmup, barrier, sampler)
    outputs = wl.last_step_outputs() if (full and args.dump_outputs) else None
    kms = wl.kernel_ms()
    t = torch.tensor([ms], device=wl.dev, dtype=torch.float64)
    per_rank = [ms]
    if world > 1:
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        per_rank = [float(x.item()) for x in g]
    ms_total = max(per_rank)
    fps = world * B * steps / (ms_total / 1e3)
    res = {"name": name, "B": B, "steps": steps, "fps": fps, "ms_total": ms_total, "per_rank_ms": per_rank, "kernel_ms": kms,
           "markers_per_frame": n_markers / (steps * B), "parity": parity, "clocks": clocks, "counters": wl.det.counters(), "wl": wl,
           "outputs": outputs}
    res["wall_ms"] = wl.wall_ms
    e2e = None
    if not args.skip_e2e:
        n_e = steps if (full or B == 1) else max(3, steps // 4)
        ms2, info = wl.time_e2e(n_e, barrier)
        t = torch.tensor([ms2], device=wl.dev, dtype=torch.float64)
        per_rank2, h2d = [ms2], [info["h2d_only_gbs"]]
        if world > 1:
            g = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(g, t)
            per_rank2 = [float(x.item()) for x in g]
            t = torch.tensor([info["h2d_only_gbs"]], device=wl.dev, dtype=torch.float64)
            dist.all_gather(g, t)
            h2d = [float(x.item()) for x in g]
        e2e_fps = world * B * n_e / (max(per_rank2) / 1e3)
        same = counts is None or info["counts"] == list(counts)
        e2e = {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": info["h2d_bytes_per_step"],
               "d2h_bytes_per_step": info["d2h_bytes_per_step"], "chunk_frames": info["chunk_frames"],
               "same_counts_as_device_path": bool(same), "per_rank_ms": per_rank2,
               # pinned H2D copies alone (same buffer, same chunking, no kernels), per rank, measured one rank after the
               # other's e2e leg but concurrently across ranks: the host-side ceiling of e2e
               "h2d_only_gbs": h2d, "h2d_gbs_in_e2e": e2e_fps * W * H / 1e9,
               # the ceiling in the same max-over-ranks convention as `value`: every rank moves the same bytes, the slowest
               # rank's link decides (on the 8-GPU boxes of this pool GPUs 0-3 and 4-7 sit behind host bridges of different speed)
               "h2d_ceiling_gbs": world * min(h2d), "frac_of_h2d_ceiling": (e2e_fps * W * H / 1e9) / max(world * min(h2d), 1e-9),
               "per_rank_frac_of_own_h2d": [B * n_e * W * H / (m / 1e3) / 1e9 / max(g, 1e-9) for m, g in zip(per_rank2, h2d)]}
    res["e2e"] = e2e
    return res


def roofline_of(res, world, peak, peak_src):
    wl, kms, B = res["wl"], res["kernel_ms"], res["B"]
    W, H = wl.W, wl.H
    dom = max(kms, key=kms.get)
    alg = algorithmic_bytes(dom, W, H, B, None)
    achieved = alg / (kms[dom] / 1e3) / 1e9
    S = oracle_params(wl.cfg).warp_size
    n_c = int(res["counters"]["candidates"])
    warp_gbs = n_c * 2.0 * S * S / (max(kms["sample"], 1e-6) / 1e3) / 1e9
    thr_gbs = 2.0 * W * H * B / (max(kms["threshold"], 1e-6) / 1e3) / 1e9
    traffic, tsrc = ncu_traffic(res["name"], dom) if B == wl.cfg["batch"] else (None, None)
    fps1 = res["fps"] / world
    return {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_unit": "dram bytes per launch (ncu --set full: %s)" % tsrc if traffic else None,
            "algorithmic_bytes_per_launch": alg, "peak_source": peak_src, "kernel_ms": kms,
            "threshold_kernel": {"achieved": thr_gbs, "frac": thr_gbs / peak},
            # the warp stage (k_homography + k_sample): N_cand * (S^2 gathered + S^2 written) algorithmic bytes
            "warp_kernel": {"achieved": warp_gbs, "frac": warp_gbs / peak, "candidates_per_batch": n_c},
            "whole_path": {"algorithmic_bytes_per_frame": 3 * W * H, "achieved": fps1 * 3 * W * H / 1e9, "frac": fps1 * 3 * W * H / 1e9 / peak}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (default: the config's)")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-others", action="store_true", help="skip the short timing of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the markers of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU arm computed: use it with --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    host_info = bind_to_gpu_numa(local)  # before torch creates threads / pinned memory
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    res = measure_config(args.config, args, rank, local, world, torch, dist, full=True)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in res.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        log("[bench] outputs of the last timed step written to %s" % args.dump_outputs)
    unbind_cpus()
    peak, peak_src = measured_peaks()
    roofline = roofline_of(res, world, peak, peak_src)
    wl = res["wl"]
    cpu = None if args.skip_cpu else wl.cpu_baselines()
    W, H, B = wl.W, wl.H, res["B"]
    n_launch = KERNELS_PER_BATCH + (1 if wl.cfg["params"].get("erosion") else 0)
    del res["wl"], wl
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, short form (1 GPU runs only) -----------------------------------------------
    others = None
    if world == 1 and not args.skip_others and args.config == "C4" and not args.batch:
        others = {}
        for name in ("C1", "C2", "C3", "C5", "C4s4", "C4r1"):
            try:
                r = measure_config(name, args, 0, local, 1, torch, dist, full=False)
                rf = roofline_of(r, 1, peak, peak_src)
                c = CONFIGS[name]
                o = {"workload": c["workload"], "frames_per_step": r["B"], "steps": r["steps"], "value": r["fps"], "unit": "frames/s",
                     "ms_per_step": r["ms_total"] / r["steps"], "mpix_per_s": r["fps"] * c["W"] * c["H"] / 1e6,
                     "markers_per_frame": r["markers_per_frame"], "parity": r["parity"],
                     "e2e": None if r["e2e"] is None else {k: r["e2e"][k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")},
                     "dominant_kernel": rf["kernel"], "roofline_frac": rf["frac"], "roofline_achieved_gbs": rf["achieved"],
                     "kernel_ms": r["kernel_ms"]}
                if not args.skip_cpu:
                    cb = r["wl"].cpu_baselines(budget_px=4e8)
                    o["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
                others[name] = o
                del r["wl"], r
                torch.cuda.empty_cache()
            except SystemExit:
                raise
            except Exception as e:  # a side measurement must not take the headline line down
                others[name] = {"error": "%s: %s" % (type(e).__name__, e)}
                log("[bench] other config %s failed: %r" % (name, e))

    line = {"metric": METRIC.get(args.config, "frames_per_s_" + args.config), "value": res["fps"], "unit": "frames/s", "n_gpus": world,
            "steps": res["steps"], "warmup": args.warmup, "ms_per_step": res["ms_total"] / res["steps"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "mpix_per_s": res["fps"] * W * H / 1e6,
            "config": config_dict(CONFIGS[args.config], B),
            "pipelining": "2 batches in flight per GPU inside ONE library context (ab_enqueue_batch_device twice before "
                          "ab_fetch_results); every step enqueues one batch and fetches its markers",
            "markers_per_frame": res["markers_per_frame"], "parity": res["parity"], "clocks": res["clocks"], "e2e": res["e2e"],
            "per_rank_ms": res["per_rank_ms"], "host": host_info,
            "gpu_launches": n_launch * res["steps"], "roofline": roofline, "cpu_baseline": cpu, "other_configs": others,
            "target_frames_per_s": 2000}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
