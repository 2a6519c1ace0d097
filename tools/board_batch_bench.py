"""Board poses for whole batches: the batch board stage (ab_set_board / ab_get_boards) against one ab_detect_board call per
frame after the batch, which is how bench.py's C2 gets board poses.

Workload: 64 seeded views of a 4x6 board (tilt <= 40 deg, noise sigma 1.5, 24 markers, 1280x720; the frames of
tests/test_board_batch.py), erosion + LINES, board pose with the synthetic camera; a batch of 256 repeats them 4 times.  Per batch
size, alternated within every repetition:
  a  ab_detect_batch, then ab_detect_board per frame       (host frames, chunks of 32)
  b  ab_detect_batch with the board armed, ab_get_boards   (host frames, chunks of 32)
  c  ab_enqueue_batch_device / ab_fetch_results with two batches in flight, board armed (c_armed) and disarmed (c_disarmed)
Prints one JSON line: frames/s per run (median, min, max over the repetitions), the board kernel's milliseconds per batch
(ab_get_kernel_ms entry 11, timing on) and the GPU's name and power limit.
    python tools/board_batch_bench.py [--reps 5] [--steps 8] [--batches 64,256]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

W, H, SIZE, SEED, CAP = 1280, 720, 0.05, 8, 64


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # the measurement itself needs the GPU; only the label is missing
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=8, help="batches per timed run")
    ap.add_argument("--batches", default="64,256")
    args = ap.parse_args()
    import torch
    from aruco_b200 import FiducidalMarkers, MarkerDetector, synth
    from aruco_b200._lib import ab_board, ab_board_config, ab_marker
    ids = [int(m["id"]) for m in json.load(open(os.path.join(ROOT, "tests", "golden", "expected.json")))["boards"]["board_pix"]["markers"]]
    img, cfg = FiducidalMarkers.createBoardImage((4, 6), 100, 20, ids)
    frames64, _ = synth.warp_board(img, cfg.objPoints, 64, W, H, seed=SEED)
    K, D = synth.camera_for(W, H)
    Kf, Df = np.ascontiguousarray(K.reshape(9)), np.ascontiguousarray(D)
    cids = np.ascontiguousarray(np.array(cfg.ids, np.int32))
    cpts = np.ascontiguousarray(cfg.objPoints.astype(np.float32).reshape(-1))
    bcfg = ab_board_config(len(cids), cfg.mInfoType, cids.ctypes.data, cpts.ctypes.data)
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    name, power = gpu_info()
    result = {"tool": "board_batch_bench", "gpu": name, "power_limit": power, "torch_device": torch.cuda.get_device_name(0),
              "workload": "4x6 board, 24 markers, 1280x720, erosion + LINES, board pose; %d reps x %d batches" % (args.reps, args.steps),
              "runs": {}}
    for B in [int(x) for x in args.batches.split(",")]:
        frames = np.ascontiguousarray(np.concatenate([frames64] * (B // 64 + 1))[:B])
        host = torch.from_numpy(frames).pin_memory()
        dev = torch.from_numpy(frames).cuda()
        torch.cuda.synchronize()
        # host frames in chunks of 32, as bench.py's end-to-end timing; the device path on a second context reserved for B
        dh, dd = MarkerDetector(0), MarkerDetector(0)
        for d in (dh, dd):
            d.enableErosion(True)
        dh.reserve(W, H, 32)
        dd.reserve(W, H, B)
        out = (ab_marker * (B * CAP))()
        cnt = (C.c_int32 * B)()
        boards, bm = (ab_board * B)(), (ab_marker * (B * CAP))()
        outm, resb = (ab_marker * CAP)(), ab_board()

        def arm(det, on):
            rc = det._lib.ab_set_board(det._h, C.byref(bcfg) if on else None, P(Kf), P(Df), SIZE, -1.0, 0)
            assert rc == 0, det._lib.ab_last_error(det._h)

        def host_batch():
            dh._check(dh._lib.ab_detect_batch(dh._h, C.c_void_p(host.data_ptr()), W, H, W, W * H, B, None, None, -1.0, out, CAP, cnt))

        def run_a(steps):
            for _ in range(steps):
                host_batch()
                for f in range(B):
                    fm = (ab_marker * CAP).from_buffer(out, f * CAP * C.sizeof(ab_marker))
                    dh._check(dh._lib.ab_detect_board(dh._h, fm, cnt[f], C.byref(bcfg), P(Kf), P(Df), SIZE, -1.0, 0, outm, C.byref(resb)))
                    assert resb.has_pose

        def run_b(steps):
            for _ in range(steps):
                host_batch()
                dh._check(dh._lib.ab_get_boards(dh._h, B, boards, bm, CAP))
                assert all(boards[f].has_pose for f in range(B))

        def enqueue():
            dd._check(dd._lib.ab_enqueue_batch_device(dd._h, C.c_void_p(dev.data_ptr()), W, H, W, W * H, B, None, None, -1.0))

        def run_c(steps):
            enqueue()
            for i in range(steps):
                if i + 1 < steps:
                    enqueue()
                dd._check(dd._lib.ab_fetch_results(dd._h, out, CAP, cnt))

        runs = {"a_per_frame_board": (dh, False, run_a), "b_batch_board": (dh, True, run_b), "c_armed": (dd, True, run_c),
                "c_disarmed": (dd, False, run_c)}
        for det, on, fn in runs.values():  # warm-up: every shape and both in-flight slots
            arm(det, on)
            fn(2)
        fps = {k: [] for k in runs}
        for rep in range(args.reps):
            for key, (det, on, fn) in runs.items():
                arm(det, on)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(args.steps)
                torch.cuda.synchronize()
                fps[key].append(B * args.steps / (time.perf_counter() - t0))  # every run ends in a fetch: the host clock is the device clock
        # board kernel time per batch: one stream, timing on
        arm(dd, True)
        dd.enable_timing(True)
        kms = []
        ms = np.zeros(12, np.float32)
        for _ in range(args.reps):
            enqueue()
            dd._check(dd._lib.ab_fetch_results(dd._h, out, CAP, cnt))
            dd._check(dd._lib.ab_get_kernel_ms(dd._h, P(ms), 12))
            kms.append(float(ms[11]))
            total = float(ms.sum())
        dd.enable_timing(False)
        result["runs"][str(B)] = {
            **{k: {"frames_per_s": round(statistics.median(v), 1), "min": round(min(v), 1), "max": round(max(v), 1)} for k, v in fps.items()},
            "board_kernel_ms_per_batch": {"median": round(statistics.median(kms), 4), "min": round(min(kms), 4), "max": round(max(kms), 4)},
            "kernels_ms_per_batch_timed": round(total, 3)}
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
