"""Seeded stereo calibration data and the comparisons of the stereo tests: correspondence sets of a 24-marker planar board seen
by two distorted cameras, the host build of the stereo arithmetic (tests/hostcheck/hostcheck_stereo.cpp), and the tolerances
against cv2.stereoCalibrateExtended (flags CALIB_FIX_INTRINSIC) on identical f32 inputs."""
import ctypes as C
import os

import numpy as np

from calib_data import board_points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DEFAULT = (3, 30, 1e-6)  # cv2's default TermCriteria(COUNT + EPS, 30, 1e-6)
CONVERGED = (3, 500, np.finfo(np.float64).eps)

# Tolerances.  Measured with cv2 4.13 on seeded sets of this generator (1-40 views, 0.05-0.5 px noise, dropped markers):
# - at CONVERGED, reversing the view order (which changes rounding only) moves cv2 by at most 6e-15 rad in R, 2.5e-14
#   relative in T and 1e-13 px in the per-view errors;
# - one f32 ulp on camera 1's image points moves the converged R by 4.5e-8..2.6e-7 rad and T by 2.3e-7..1.3e-6 relative;
# - at DEFAULT cv2 stops before convergence: reversing the view order moves it by up to 2.8e-9 rad in R, 2.6e-8 in T,
#   5.9e-8 in rms and 1.4e-5 px in the per-view errors.
# The default tolerances cover ~3x cv2's own stop-rule spread.  At CONVERGED the host build agrees with cv2 to ~1e-13 on
# most sets, but near the minimum a step that lowers |e|^2 by less than its rounding is accepted by one implementation and
# rejected by the other: on seed 0 cv2 takes one more step of 3.1e-10 rad in R (2e-9 relative in T, 2.1e-9 px in the
# per-view errors).  The converged tolerances allow ~3x that and stay ~100x below the data's 1-ulp sensitivity.
TOL = {
    "converged": {"R_rad": 1e-9, "T_rel": 1e-8, "rms_rel": 1e-11, "pve_px": 1e-8, "EF_rel": 1e-8, "reproj_px": 1e-6},
    "default": {"R_rad": 1e-8, "T_rel": 1e-7, "rms_rel": 2e-7, "pve_px": 1e-4, "EF_rel": 1e-7, "reproj_px": 1e-3},
}


def random_camera(rng, W, H):
    f = rng.uniform(0.75, 1.1) * W
    K = np.array([[f, 0, W / 2 + rng.uniform(-20, 20)], [0, f * rng.uniform(0.98, 1.02), H / 2 + rng.uniform(-15, 15)], [0, 0, 1]])
    D = np.array([rng.uniform(-0.3, 0.1), rng.uniform(-0.05, 0.12), rng.uniform(-2e-3, 2e-3), rng.uniform(-2e-3, 2e-3),
                  rng.uniform(-0.03, 0.01)])
    return K, D


def make_stereo_views(seed, n_views=20, W=1280, H=720, sigma=0.15, drop=0.15, baseline="x", rot=0.15):
    """n_views seeded views of board_points() seen by two seeded distorted cameras.  Camera 2 sits at a baseline of 6-15 cm
    along x (or y) from camera 1, turned towards camera 1's axis at the mean board distance plus a rotation ~ N(0, rot) rad
    per axis; every board corner lies 20 px inside both
    frames; image noise sigma px; each marker is dropped with probability `drop` (from both cameras).  Returns a dict with
    W, H, objs, imgs1, imgs2, K1, D1, K2, D2 and the truth R, T."""
    import cv2
    rng = np.random.default_rng(seed)
    K1, D1 = random_camera(rng, W, H)
    K2, D2 = random_camera(rng, W, H)
    b = rng.uniform(-0.15, -0.06)
    T = np.array([b, rng.uniform(-0.01, 0.01), rng.uniform(-0.01, 0.01)])
    if baseline == "y":
        T = T[[1, 0, 2]]
    z0 = 0.55 * max(K1[0, 0], K2[0, 0]) / 1000  # mean board distance: about 580 px board height
    toe = np.array([T[1], -T[0], 0.0]) / z0
    R, _ = cv2.Rodrigues(toe + rng.normal(0, rot, 3))
    obj = board_points()
    objs, imgs1, imgs2 = [], [], []
    for _ in range(n_views):
        for _ in range(5000):
            rv = rng.normal(0, 0.3, 3)
            tv = np.array([rng.uniform(-0.05, 0.05) - T[0] / 2, rng.uniform(-0.03, 0.03) - T[1] / 2, z0 * rng.uniform(0.85, 1.15)])
            R0, _ = cv2.Rodrigues(rv)
            rv2, _ = cv2.Rodrigues(R @ R0)
            t2 = R @ tv + T
            if t2[2] < 0.2:
                continue
            p1 = cv2.projectPoints(obj.astype(np.float64), rv, tv, K1, D1)[0].reshape(-1, 2)
            p2 = cv2.projectPoints(obj.astype(np.float64), rv2, t2, K2, D2)[0].reshape(-1, 2)
            if all(((p[:, 0] > 20) & (p[:, 0] < W - 20) & (p[:, 1] > 20) & (p[:, 1] < H - 20)).all() for p in (p1, p2)):
                break
        else:
            raise RuntimeError("make_stereo_views: no pose fits both frames")
        keep = np.repeat(rng.random(len(obj) // 4) > drop, 4)
        if keep.sum() < 8:
            keep[:8] = True
        objs.append(np.ascontiguousarray(obj[keep]))
        imgs1.append(np.ascontiguousarray((p1 + rng.normal(0, sigma, p1.shape))[keep].astype(np.float32)))
        imgs2.append(np.ascontiguousarray((p2 + rng.normal(0, sigma, p2.shape))[keep].astype(np.float32)))
    return {"W": W, "H": H, "objs": objs, "imgs1": imgs1, "imgs2": imgs2, "K1": K1, "D1": D1, "K2": K2, "D2": D2, "R": R, "T": T}


# (seed, n_views, sigma, drop, baseline, relative rotation sigma): 12 sets
CASES = [(0, 25, 0.15, 0.15, "x", 0.05), (1, 5, 0.1, 0.0, "x", 0.03), (2, 1, 0.15, 0.0, "x", 0.03), (3, 40, 0.5, 0.2, "x", 0.05),
         (4, 12, 0.05, 0.3, "y", 0.05), (5, 8, 0.3, 0.1, "y", 0.03), (6, 30, 0.15, 0.15, "x", 0.08), (7, 20, 0.3, 0.25, "y", 0.08),
         (8, 15, 0.15, 0.15, "x", 0.1), (9, 35, 0.2, 0.3, "y", 0.1), (10, 6, 0.15, 0.0, "x", 0.02), (11, 2, 0.2, 0.1, "y", 0.05)]


def case(c):
    seed, n, sigma, drop, baseline, rot = c
    return make_stereo_views(seed, n_views=n, sigma=sigma, drop=drop, baseline=baseline, rot=rot)


_hc = None


class ab_stereo_result(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("T", C.c_double * 3), ("E", C.c_double * 9), ("F", C.c_double * 9), ("rms", C.c_double),
                ("iterations", C.c_int32), ("status", C.c_int32)]


def hostcheck():
    global _hc
    if _hc is None:
        lib = C.CDLL(os.path.join(ROOT, "tests", "_build", "libhostcheck_stereo.so"))
        lib.hc_stereo_calibrate.restype = C.c_int
        lib.hc_stereo_calibrate.argtypes = [C.c_int] + [C.c_void_p] * 8 + [C.c_int, C.c_double] + [C.c_void_p] * 4
        _hc = lib
    return _hc


def _stack(views, dim):
    return np.ascontiguousarray(np.concatenate([np.asarray(v, np.float32).reshape(-1, dim) for v in views]) if len(views)
                                else np.zeros((0, dim), np.float32))


def _d5(D):
    return np.zeros(5) if D is None else np.concatenate([np.asarray(D, np.float64).ravel(), np.zeros(5)])[:5]


def host_stereo(objs, imgs1, imgs2, K1, D1, K2, D2, criteria=DEFAULT):
    """The host build of k_stereo_calibrate's arithmetic on one pair: (status, {rms, R, T, E, F, rvecs, tvecs, pve, iterations})."""
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    n = np.array([len(o) for o in objs], np.int32)
    obj, i1, i2 = _stack(objs, 3), _stack(imgs1, 2), _stack(imgs2, 2)
    k1, k2 = np.ascontiguousarray(K1, np.float64).reshape(9), np.ascontiguousarray(K2, np.float64).reshape(9)
    d1, d2 = _d5(D1), _d5(D2)
    nv = max(len(objs), 1)
    rv, tv, pve = np.zeros((nv, 3)), np.zeros((nv, 3)), np.zeros((nv, 2))
    r = ab_stereo_result()
    st = hostcheck().hc_stereo_calibrate(len(objs), P(n), P(obj), P(i1), P(i2), P(k1), P(d1), P(k2), P(d2), int(criteria[1]),
                                         float(criteria[2]), C.addressof(r), P(rv), P(tv), P(pve))
    m = lambda a: np.array(a, np.float64).reshape(3, 3)
    return st, {"rms": float(r.rms), "R": m(r.R), "T": np.array(r.T, np.float64), "E": m(r.E), "F": m(r.F), "rvecs": rv[:len(objs)],
                "tvecs": tv[:len(objs)], "pve": pve[:len(objs)], "iterations": int(r.iterations)}


def cv2_stereo(d, criteria=DEFAULT):
    import cv2
    r = cv2.stereoCalibrateExtended(d["objs"], d["imgs1"], d["imgs2"], d["K1"], d["D1"], d["K2"], d["D2"], (d["W"], d["H"]), None, None,
                                    flags=cv2.CALIB_FIX_INTRINSIC, criteria=criteria)
    return {"rms": r[0], "R": r[5], "T": r[6].ravel(), "E": r[7], "F": r[8], "rvecs": [x.ravel() for x in r[9]],
            "tvecs": [x.ravel() for x in r[10]], "pve": np.asarray(r[11]).reshape(-1, 2)}


def rot_angle(Ra, Rb):
    M = np.asarray(Ra).T @ np.asarray(Rb)
    return 0.5 * float(np.linalg.norm([M[2, 1] - M[1, 2], M[0, 2] - M[2, 0], M[1, 0] - M[0, 1]]))


def compare(got, ref, d, level, what=""):
    """Asserts the `level` tolerances between two solutions; returns the measured maxima."""
    import cv2
    tol = TOL[level]
    tn = float(np.linalg.norm(ref["T"]))
    m = {"R_rad": rot_angle(got["R"], ref["R"]), "T_rel": float(np.linalg.norm(np.ravel(got["T"]) - np.ravel(ref["T"]))) / tn,
         "rms_rel": abs(got["rms"] - ref["rms"]) / ref["rms"],
         "pve_px": float(np.abs(np.asarray(got["pve"]).reshape(-1, 2) - np.asarray(ref["pve"]).reshape(-1, 2)).max()),
         "EF_rel": max(float(np.abs(np.asarray(got[k]) - np.asarray(ref[k])).max() / np.abs(ref[k]).max()) for k in ("E", "F"))}
    rep = 0.0
    for o, rg, tg, rr, tr in zip(d["objs"], got["rvecs"], got["tvecs"], ref["rvecs"], ref["tvecs"]):
        pg = cv2.projectPoints(o.astype(np.float64), np.ravel(rg), np.ravel(tg), d["K1"], d["D1"])[0]
        pr = cv2.projectPoints(o.astype(np.float64), np.ravel(rr), np.ravel(tr), d["K1"], d["D1"])[0]
        rep = max(rep, float(np.abs(pg - pr).max()))
    m["reproj_px"] = rep
    bad = {k: v for k, v in m.items() if not v <= tol[k]}
    assert not bad, "%s (%s): %s exceed %s" % (what, level, bad, tol)
    return m
