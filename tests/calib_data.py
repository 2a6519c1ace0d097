"""Seeded calibration data and the comparisons of the calibration tests: correspondence sets of a 24-marker planar board seen
by a distorted camera, the host build of the calibration arithmetic (tests/hostcheck/hostcheck_calib.cpp), and the tolerances
against cv2.calibrateCamera on identical f32 inputs."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Tolerances against cv2 (identical f32 inputs).  cv2 converges onto the minimum on such data: refitting its answer with an
# independent tight LM moves K by < 1e-12 relative and k3 by ~1e-8, while one f32 ulp on the image points moves k3 by up
# to 3.4e-4 -- so the tolerances below are far inside the data's own sensitivity but well outside the optimiser's.
K_RTOL = 1e-7
D_ATOL = 1e-5
RMS_RTOL = 1e-9
REPROJ_ATOL = 1e-4  # px, every calibration point under each solution with its own extrinsics


def board_points(rows=6, cols=4, side=0.04, gap=0.01):
    """4 corners per marker of a rows x cols marker board (metres, z = 0, centred)."""
    obj = []
    for r in range(rows):
        for c in range(cols):
            x0, y0 = c * (side + gap), r * (side + gap)
            obj += [[x0, y0, 0], [x0 + side, y0, 0], [x0 + side, y0 + side, 0], [x0, y0 + side, 0]]
    obj = np.array(obj, np.float64)
    obj[:, :2] -= obj[:, :2].mean(0)
    return obj.astype(np.float32)


def make_views(seed, n_views=25, W=1280, H=720, sigma=0.15, drop=0.15, K=None, D=None, tilt=0.35):
    """n_views seeded views of board_points(): camera K / D (drawn from the seed when None), pose tilts ~ N(0, tilt) rad,
    image noise sigma px, each marker dropped with probability `drop`.  Returns (W, H, objs, imgs) as cv2 takes them."""
    import cv2
    rng = np.random.default_rng(seed)
    if K is None:
        f = rng.uniform(0.75, 1.1) * W
        K = np.array([[f, 0, W / 2 + rng.uniform(-20, 20)], [0, f * rng.uniform(0.98, 1.02), H / 2 + rng.uniform(-15, 15)], [0, 0, 1]])
    if D is None:
        D = np.array([rng.uniform(-0.3, 0.1), rng.uniform(-0.05, 0.12), rng.uniform(-2e-3, 2e-3), rng.uniform(-2e-3, 2e-3),
                      rng.uniform(-0.03, 0.01)])
    obj = board_points()
    objs, imgs = [], []
    for _ in range(n_views):
        for _ in range(1000):
            rv = rng.normal(0, tilt, 3)
            tv = np.array([rng.uniform(-0.05, 0.05), rng.uniform(-0.03, 0.03), rng.uniform(0.35, 0.6)]) * K[0, 0] / 1100
            p, _ = cv2.projectPoints(obj.astype(np.float64), rv, tv, K, D)
            p = p.reshape(-1, 2)
            if (p[:, 0] > 20).all() and (p[:, 0] < W - 20).all() and (p[:, 1] > 20).all() and (p[:, 1] < H - 20).all():
                break
        keep = np.repeat(rng.random(len(obj) // 4) > drop, 4)
        if keep.sum() < 8:
            keep[:8] = True
        objs.append(np.ascontiguousarray(obj[keep]))
        imgs.append(np.ascontiguousarray((p + rng.normal(0, sigma, p.shape))[keep].astype(np.float32)))
    return W, H, objs, imgs


_hc = None


def hostcheck():
    global _hc
    if _hc is None:
        lib = C.CDLL(os.path.join(ROOT, "tests", "_build", "libhostcheck_calib.so"))
        lib.hc_calibrate.restype = C.c_int
        lib.hc_calibrate.argtypes = [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 9
        _hc = lib
    return _hc


def host_calibrate(W, H, objs, imgs):
    """The host build of k_calibrate's arithmetic on one camera: (status, {rms, K, D, rvecs, tvecs, iterations})."""
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    n = np.array([len(o) for o in objs], np.int32)
    obj = np.ascontiguousarray(np.concatenate([np.asarray(o, np.float32).reshape(-1, 3) for o in objs]) if len(objs) else np.zeros((0, 3), np.float32))
    img = np.ascontiguousarray(np.concatenate([np.asarray(i, np.float32).reshape(-1, 2) for i in imgs]) if len(imgs) else np.zeros((0, 2), np.float32))
    K, D, rms, it = np.zeros(9), np.zeros(5), np.zeros(1), np.zeros(1, np.int32)
    rv, tv = np.zeros((max(len(objs), 1), 3)), np.zeros((max(len(objs), 1), 3))
    st = hostcheck().hc_calibrate(W, H, len(objs), P(n), P(obj), P(img), P(K), P(D), P(rms), P(it), P(rv), P(tv))
    return st, {"rms": float(rms[0]), "K": K.reshape(3, 3), "D": D, "rvecs": rv[:len(objs)], "tvecs": tv[:len(objs)],
                "iterations": int(it[0])}


def reprojections(objs, K, D, rvecs, tvecs):
    import cv2
    return [cv2.projectPoints(np.asarray(o, np.float64), np.asarray(r, np.float64).reshape(3), np.asarray(t, np.float64).reshape(3),
                              np.asarray(K, np.float64), np.asarray(D, np.float64).ravel())[0].reshape(-1, 2)
            for o, r, t in zip(objs, rvecs, tvecs)]


def compare(got, ref, objs, what=""):
    """Asserts the tolerances between two solutions {rms, K, D, rvecs, tvecs}; returns the measured maxima."""
    Kg, Kr = np.asarray(got["K"], np.float64), np.asarray(ref["K"], np.float64)
    k_rel = float(max(abs(Kg[i, j] - Kr[i, j]) / abs(Kr[i, j]) for i, j in ((0, 0), (1, 1), (0, 2), (1, 2))))
    d_abs = float(np.abs(np.asarray(got["D"], np.float64).ravel()[:5] - np.asarray(ref["D"], np.float64).ravel()[:5]).max())
    rms_rel = abs(got["rms"] - ref["rms"]) / ref["rms"]
    pg = reprojections(objs, got["K"], got["D"], got["rvecs"], got["tvecs"])
    pr = reprojections(objs, ref["K"], ref["D"], ref["rvecs"], ref["tvecs"])
    rep = float(max(np.abs(a - b).max() for a, b in zip(pg, pr)))
    m = {"K_rel": k_rel, "D_abs": d_abs, "rms_rel": rms_rel, "reproj_px": rep}
    assert k_rel <= K_RTOL and d_abs <= D_ATOL and rms_rel <= RMS_RTOL and rep <= REPROJ_ATOL, "%s: %s" % (what, m)
    return m


def cv2_calibrate(W, H, objs, imgs):
    import cv2
    rms, K, D, rv, tv = cv2.calibrateCamera([np.asarray(o, np.float32) for o in objs], [np.asarray(i, np.float32) for i in imgs], (W, H),
                                            None, None)
    return {"rms": rms, "K": K, "D": D.ravel(), "rvecs": [r.ravel() for r in rv], "tvecs": [t.ravel() for t in tv]}


# (seed, n_views, sigma, drop): 12 sets -- varied K and distortion from the seed, 5..40 views
CASES = [(0, 25, 0.15, 0.15), (1, 25, 0.15, 0.15), (2, 5, 0.1, 0.0), (3, 8, 0.2, 0.2), (4, 12, 0.15, 0.15), (5, 40, 0.15, 0.15),
         (6, 30, 0.3, 0.1), (7, 20, 0.05, 0.25), (8, 15, 0.15, 0.15), (9, 35, 0.15, 0.3), (10, 6, 0.15, 0.0), (11, 25, 0.5, 0.15)]
