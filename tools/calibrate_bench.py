"""Camera calibration throughput: ab_calibrate_cameras (k_calibrate, one CTA per camera) against cv2.calibrateCamera on the host.

Each camera has 30 views x 96 points (a 24-marker board, seeded poses, distortion, 0.15 px noise).  For 1, 16, 148 and 1024
cameras per call it reports the median device time per call (host clock around the synchronising call, after warm-up) and
cv2's time for the same cameras with one thread and with all threads; the card's name and power limit are read in the same run.
Prints one JSON line; --out also writes it to a file.

    python tools/calibrate_bench.py [--reps 5] [--cv2-cams 16] [--out /tmp/calibrate_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cv2-cams", type=int, default=16, help="cameras cv2 is timed on; its per-camera time is scaled to each size")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import cv2
    from calib_data import make_views
    from aruco_b200 import MarkerDetector, calibrateCameras
    det = MarkerDetector(0)
    # 64 distinct seeded cameras, repeated to fill the larger calls; all drop=0 so every view has 96 points
    base = [make_views(s, n_views=30, drop=0.0) for s in range(64)]
    cams = [(o, i, (W, H)) for W, H, o, i in base]
    sizes = [1, 16, 148, 1024]
    rows = []
    nthreads = cv2.getNumThreads()
    cv2_t = {}
    for threads in (1, nthreads):
        cv2.setNumThreads(threads)
        t0 = time.perf_counter()
        for W, H, o, i in base[:a.cv2_cams]:
            cv2.calibrateCamera(o, i, (W, H), None, None)
        cv2_t[threads] = (time.perf_counter() - t0) / a.cv2_cams
    cv2.setNumThreads(nthreads)
    for n in sizes:
        batch = [cams[k % len(cams)] for k in range(n)]
        res = calibrateCameras(batch, detector=det)  # warm-up (module load, scratch growth)
        assert all(r is not None for r in res)
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            calibrateCameras(batch, detector=det)
            ts.append(time.perf_counter() - t0)
        ms = float(np.median(ts)) * 1e3
        rows.append({"cameras": n, "views": 30, "points_per_view": 96, "device_ms_per_call": round(ms, 3),
                     "device_ms_per_camera": round(ms / n, 4), "cv2_1thread_ms": round(cv2_t[1] * n * 1e3, 1),
                     "cv2_%dthreads_ms" % nthreads: round(cv2_t[nthreads] * n * 1e3, 1)})
    out = {"card": card(), "cv2_threads": nthreads, "cv2_ms_per_camera_1thread": round(cv2_t[1] * 1e3, 2),
           "cv2_ms_per_camera_all_threads": round(cv2_t[nthreads] * 1e3, 2), "reps": a.reps, "rows": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
