"""Stereo calibration throughput: ab_stereo_calibrate (k_stereo_calibrate, one CTA per camera pair) against cv2.stereoCalibrate
(CALIB_FIX_INTRINSIC) on the host.

Each pair has 30 views x 96 points (a 24-marker board seen by two distorted cameras, seeded poses, 0.15 px noise) and runs with
cv2's default criteria (30, 1e-6).  For 1, 16, 148 and 1024 pairs per call it reports the median device time per call (host
clock around the synchronising call, after warm-up) and cv2's time for the same pairs with one thread and with all threads
(timed on --cv2-pairs pairs and scaled); the card's name and power limit are read in the same run.  Prints one JSON line; --out
also writes it to a file.

    python tools/stereo_calibrate_bench.py [--reps 5] [--cv2-pairs 16] [--out /tmp/stereo_calibrate_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cv2-pairs", type=int, default=16, help="pairs cv2 is timed on; its per-pair time is scaled to each size")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import cv2
    from calibrate_bench import card
    from stereo_data import make_stereo_views
    from aruco_b200 import MarkerDetector, stereoCalibratePairs
    det = MarkerDetector(0)
    # 64 distinct seeded pairs, repeated to fill the larger calls; all drop=0 so every view has 96 points
    base = [make_stereo_views(s, n_views=30, drop=0.0, rot=0.05) for s in range(64)]
    pairs = [(d["objs"], d["imgs1"], d["imgs2"], d["K1"], d["D1"], d["K2"], d["D2"]) for d in base]
    nthreads = cv2.getNumThreads()
    cv2_t = {}
    for threads in (1, nthreads):
        cv2.setNumThreads(threads)
        t0 = time.perf_counter()
        for d in base[:a.cv2_pairs]:
            cv2.stereoCalibrate(d["objs"], d["imgs1"], d["imgs2"], d["K1"], d["D1"], d["K2"], d["D2"], (d["W"], d["H"]),
                                flags=cv2.CALIB_FIX_INTRINSIC)
        cv2_t[threads] = (time.perf_counter() - t0) / a.cv2_pairs
    cv2.setNumThreads(nthreads)
    rows = []
    for n in [1, 16, 148, 1024]:
        batch = [pairs[k % len(pairs)] for k in range(n)]
        res = stereoCalibratePairs(batch, detector=det)  # warm-up (module load, scratch growth)
        assert all(r is not None for r in res)
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            stereoCalibratePairs(batch, detector=det)
            ts.append(time.perf_counter() - t0)
        ms = float(np.median(ts)) * 1e3
        rows.append({"pairs": n, "views": 30, "points_per_view": 96, "device_ms_per_call": round(ms, 3), "device_ms_per_pair": round(ms / n, 4),
                     "cv2_1thread_ms": round(cv2_t[1] * n * 1e3, 1), "cv2_%dthreads_ms" % nthreads: round(cv2_t[nthreads] * n * 1e3, 1)})
    out = {"card": card(), "cv2_threads": nthreads, "cv2_ms_per_pair_1thread": round(cv2_t[1] * 1e3, 2),
           "cv2_ms_per_pair_all_threads": round(cv2_t[nthreads] * 1e3, 2), "reps": a.reps, "rows": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
