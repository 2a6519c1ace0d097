"""ab_stereo_calibrate / aruco_b200.stereoCalibrate* on the device (k_stereo_calibrate): equal to the host build of the same
arithmetic and to cv2.stereoCalibrateExtended (CALIB_FIX_INTRINSIC) on identical f32 inputs, independent of the pairs sharing a
launch, bit-identical from run to run, degenerate pairs inside a call, its error returns, and end to end from rendered
stereo frames through detect_batch, per-camera calibration and the C++ driver."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, needs_cv2
from stereo_data import CASES, CONVERGED, DEFAULT, case, compare, cv2_stereo, host_stereo

pytestmark = [pytest.mark.gpu, needs_cv2]


@pytest.fixture(scope="module")
def det(built):
    from aruco_b200 import MarkerDetector
    return MarkerDetector(0)


@pytest.fixture(scope="module")
def sets():
    return [case(c) for c in CASES]


def _pair(d):
    return (d["objs"], d["imgs1"], d["imgs2"], d["K1"], d["D1"], d["K2"], d["D2"])


def as_dict(r):
    rms, K1, D1, K2, D2, R, T, E, F, rv, tv, pve = r
    return {"rms": rms, "R": R, "T": T.ravel(), "E": E, "F": F, "rvecs": [x.ravel() for x in rv], "tvecs": [x.ravel() for x in tv],
            "pve": pve}


@pytest.mark.parametrize("level", ["default", "converged"])
def test_device_matches_host_build_and_cv2(det, sets, level):
    from aruco_b200 import stereoCalibratePairs
    crit = DEFAULT if level == "default" else CONVERGED
    res = stereoCalibratePairs([_pair(d) for d in sets], criteria=crit, detector=det)
    worst = {}
    for d, r, c in zip(sets, res, CASES):
        assert r is not None, c
        assert r[5].shape == (3, 3) and r[6].shape == (3, 1) and r[11].shape == (len(d["objs"]), 2) and isinstance(r[0], float)
        st, hc = host_stereo(*_pair(d), criteria=crit)
        assert st == 0
        # the device and the host build differ only in the order of the warp sums: converged tolerances against the host at
        # both criteria levels
        for ref, name, lvl in ((hc, "host build", "converged"), (cv2_stereo(d, crit), "cv2", level)):
            for k, v in compare(as_dict(r), ref, d, lvl, "case %s vs %s" % (c, name)).items():
                worst[(name, k)] = max(worst.get((name, k), 0.0), v)
    print(level, "stereo maxima:", {"%s %s" % k: "%.3g" % v for k, v in sorted(worst.items())})


def _bits(r):
    return None if r is None else b"".join(np.ascontiguousarray(x).tobytes() for x in (np.float64(r[0]),) + r[5:9] + (np.concatenate(r[9]),
                                                                                                                    np.concatenate(r[10]), r[11]))


def test_launch_composition_and_repeat_are_bit_identical(det, sets):
    from aruco_b200 import stereoCalibratePairs
    pairs = [_pair(d) for d in sets]
    alone = [_bits(stereoCalibratePairs([p], detector=det)[0]) for p in pairs]
    assert [_bits(r) for r in stereoCalibratePairs(pairs[:1], detector=det)] == alone[:1]
    assert [_bits(r) for r in stereoCalibratePairs(pairs[3:10], detector=det)] == alone[3:10]
    order = [(7 * k + 3) % len(pairs) for k in range(300)]
    assert [_bits(r) for r in stereoCalibratePairs([pairs[j] for j in order], detector=det)] == [alone[j] for j in order]
    assert [_bits(r) for r in stereoCalibratePairs([pairs[j] for j in order], detector=det)] == [alone[j] for j in order]


def test_degenerate_pair_does_not_fail_the_call(det, sets):
    from aruco_b200 import ArucoError, stereoCalibrate, stereoCalibratePairs
    objs, i1, i2, K1, D1, K2, D2 = _pair(sets[0])
    bent = [o.copy() for o in objs]
    bent[0][:, 2] = np.linspace(0, 0.01, len(bent[0]), dtype=np.float32)
    res = stereoCalibratePairs([(objs, i1, i2, K1, D1, K2, D2), (bent, i1, i2, K1, D1, K2, D2), ([], [], [], K1, D1, K2, D2),
                                ([objs[0][:3]], [i1[0][:3]], [i2[0][:3]], K1, D1, K2, D2), (objs, i1, i2, K1, D1, K2, D2)], detector=det)
    assert res[1] is None and res[2] is None and res[3] is None
    assert _bits(res[0]) == _bits(res[4]) == _bits(stereoCalibratePairs([(objs, i1, i2, K1, D1, K2, D2)], detector=det)[0])
    with pytest.raises(ArucoError):
        stereoCalibrate(bent, i1, i2, K1, D1, K2, D2, None, detector=det)
    with pytest.raises(ArucoError):
        stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, flags=0, detector=det)
    for typ in (1, 2):  # COUNT or EPS alone
        with pytest.raises(ArucoError):
            stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, criteria=(typ, 30, 1e-6), detector=det)
    # 4 coefficients mean k3 = 0, None means no distortion
    r4 = stereoCalibratePairs([(objs, i1, i2, K1, np.r_[D1[:4], 0], K2, D2[:4]), (objs, i1, i2, K1, D1[:4], K2, np.r_[D2[:4], 0.0])],
                              detector=det)
    assert _bits(r4[0]) == _bits(r4[1])
    r0 = stereoCalibratePairs([(objs, i1, i2, K1, None, K2, None), (objs, i1, i2, K1, np.zeros(5), K2, np.zeros(5))], detector=det)
    assert _bits(r0[0]) == _bits(r0[1])


def test_error_returns(det, sets):
    import torch
    from aruco_b200 import ArucoError, MarkerDetector, _lib, stereoCalibrate
    from aruco_b200._lib import ab_stereo_pair, ab_stereo_result
    from aruco_b200.synth import render_frame
    lib, h = det._lib, det._h
    objs, i1, i2, K1, D1, K2, D2 = _pair(sets[0])
    n = np.array([len(o) for o in objs], np.int32)
    obj, a, b = (np.ascontiguousarray(np.concatenate(x)) for x in (objs, i1, i2))
    dv = lambda x, k: (C.c_double * k)(*np.ravel(x))

    def pair(nv=len(objs), np_=n.ctypes.data, o=obj.ctypes.data, p1=a.ctypes.data, p2=b.ctypes.data, k1=K1, k2=K2):
        return ab_stereo_pair(0, 0, nv, np_, o, p1, p2, dv(k1, 9), dv(D1, 5), dv(k2, 9), dv(D2, 5))
    out = ab_stereo_result()
    call = lambda p, n_=1, it=30, eps=1e-6, o=C.byref(out): lib.ab_stereo_calibrate(h, n_, C.byref(p) if p is not None else None, it, eps, o,
                                                                                     None, None, None)
    assert call(pair()) == 0 and out.status == 0
    assert call(None) == _lib.AB_E_INVALID
    assert call(pair(), o=None) == _lib.AB_E_INVALID
    assert call(pair(), n_=-1) == _lib.AB_E_INVALID
    assert call(pair(), n_=65537) == _lib.AB_E_INVALID and b"65536" in lib.ab_last_error(h)
    for it, eps in ((0, 1e-6), (1001, 1e-6), (30, -1.0), (30, float("nan")), (30, float("inf"))):
        assert call(pair(), it=it, eps=eps) == _lib.AB_E_INVALID
    bad_k = [K1 * np.array([[0, 1, 1], [1, 1, 1], [1, 1, 1]]), K1 * np.array([[1, 1, 1], [1, -1, 1], [1, 1, 1]]), np.where(np.eye(3) > 0, np.nan, K1)]
    for k in bad_k:
        assert call(pair(k1=k)) == _lib.AB_E_INVALID and b"pair 0" in lib.ab_last_error(h)
        assert call(pair(k2=k)) == _lib.AB_E_INVALID
    for p in (pair(nv=-1), pair(nv=1025), pair(np_=None), pair(o=None), pair(p1=None), pair(p2=None)):
        assert call(p) == _lib.AB_E_INVALID
    big = np.array([4097], np.int32)
    assert call(pair(nv=1, np_=big.ctypes.data)) == _lib.AB_E_INVALID
    assert lib.ab_stereo_calibrate(h, 0, None, 30, 1e-6, None, None, None, None) == 0
    # a batch in flight
    md = MarkerDetector(0)
    grey, _ = render_frame(640, 480, 4, seed=1)
    dev = torch.from_numpy(grey).cuda()
    torch.cuda.synchronize()
    md.enqueue_device(dev.data_ptr(), 640, 480, 1)
    with pytest.raises(ArucoError) as e:
        stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, detector=md)
    assert e.value.code == _lib.AB_E_STATE
    md.fetch(1)
    r = stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, detector=md)
    ref = stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, detector=det)
    assert all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(r, ref))


# ---- end to end: rendered stereo frames -> detect_batch -> calibrate per camera -> stereoCalibrate, and the C++ driver --------
# Camera 2 relative to camera 1 in warp_board_stereo's board-pixel units: a 180 px (9 cm at 0.5 mm per board pixel) baseline
# along -x, turned 0.1 rad about y towards the board.
E2E_RVEC, E2E_T = np.array([0.0, 0.1, 0.0]), np.array([-180.0, 0.0, 0.0])
# bounds against the rendering truth: measured on a B200 0.020 degrees and 1.2 % of |T| (DESIGN 8b)
E2E_MAX_DEG, E2E_MAX_T_REL = 0.05, 0.02


@pytest.fixture(scope="module")
def stereo_views(built):
    import cv2
    from aruco_b200 import FiducidalMarkers
    from aruco_b200.synth import warp_board_stereo
    img, bc = FiducidalMarkers.createBoardImage((4, 6), 100, 20, list(range(24)))
    W, H = 1280, 720
    R_lr = cv2.Rodrigues(E2E_RVEC)[0]
    f1, f2, _ = warp_board_stereo(img, bc.objPoints, 30, W, H, 5, R_lr, E2E_T)
    return W, H, f1, f2, bc, R_lr


def _save_board_config(bc, path):
    lines = ["%YAML:1.0", "---", "aruco_bc_nmarkers: %d" % bc.size(), "aruco_bc_mInfoType: %d" % bc.mInfoType, "aruco_bc_markers:"]
    for i, c in zip(bc.ids, bc.objPoints):
        pts = ", ".join("[ %r, %r, %r ]" % tuple(float(v) for v in p) for p in c)
        lines.append("   - { id:%d, corners:[ %s ] }" % (i, pts))
    path.write_text("\n".join(lines) + "\n")


def _save_camera(K, D, W, H, path):
    f = lambda a: ", ".join("%.9g" % float(v) for v in np.asarray(a, np.float32).ravel())
    path.write_text("%%YAML:1.0\n---\nimage_width: %d\nimage_height: %d\ncamera_matrix: !!opencv-matrix\n   rows: 3\n   cols: 3\n"
                    "   dt: d\n   data: [ %s ]\ndistortion_coefficients: !!opencv-matrix\n   rows: 1\n   cols: 5\n   dt: d\n"
                    "   data: [ %s ]\n" % (W, H, f(K), f(D)))


def test_end_to_end_from_rendered_stereo_views(stereo_views, tmp_path):
    import cv2
    from aruco_b200 import BoardDetector, MarkerDetector, stereoCalibrate, stereoCalibrateExtended
    W, H, f1, f2, bc, R_lr = stereo_views
    md = MarkerDetector(0)
    md.setCornerRefinementMethod(MarkerDetector.SUBPIX)  # as the C++ drivers
    bd = BoardDetector(detector=md)
    bd.setParams(bc, None, None, 0.05)
    r1, r2 = bd.detect_batch(f1), bd.detect_batch(f2)
    c1, c2 = bd.calibrate(r1, (W, H)), bd.calibrate(r2, (W, H))
    (res, objs, i1, i2) = bd.stereoCalibrate(r1, r2, c1[1], c1[2], c2[1], c2[2], raw=True, criteria=CONVERGED)
    assert len(objs) >= 20 and all(o.dtype == np.float32 for o in objs)
    assert all(np.array_equal(a, b) for a, b in zip(sum(BoardDetector.stack_stereo_views(r1, r2, bc, 0.05), []), objs + i1 + i2))
    ext = stereoCalibrateExtended(objs, i1, i2, c1[1], c1[2], c2[1], c2[2], (W, H), criteria=CONVERGED, detector=md)
    assert all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(ext[:9], res))
    d = {"W": W, "H": H, "objs": objs, "imgs1": i1, "imgs2": i2, "K1": c1[1], "D1": c1[2], "K2": c2[1], "D2": c2[2]}
    m = compare(as_dict(ext), cv2_stereo(d, CONVERGED), d, "converged", "end to end")
    # against the rendering truth: metres per board pixel from the configuration, as stack_views scales
    c = bc.objPoints[0].astype(np.float64)
    mpp = float(np.float32(0.05)) / float(np.linalg.norm(c[0] - c[1]))
    T_true = E2E_T * mpp
    ang = np.degrees(np.linalg.norm(cv2.Rodrigues(res[5].T @ R_lr)[0]))
    t_rel = float(np.linalg.norm(res[6].ravel() - T_true) / np.linalg.norm(T_true))
    print("end to end: views %d rms %.4f  vs cv2 %s  vs truth: R %.4f deg, T %.4f of |T|" % (len(objs), res[0], m, ang, t_rel))
    assert ang < E2E_MAX_DEG and t_rel < E2E_MAX_T_REL
    # the C++ driver on the same frames, with the intrinsics as its YAML carries them (f32)
    raw1, raw2, byml, cam1, cam2, out = (tmp_path / n for n in ("f1.raw", "f2.raw", "board.yml", "cam1.yml", "cam2.yml", "stereo.yml"))
    raw1.write_bytes(np.ascontiguousarray(f1).tobytes())
    raw2.write_bytes(np.ascontiguousarray(f2).tobytes())
    _save_board_config(bc, byml)
    _save_camera(c1[1], c1[2], W, H, cam1)
    _save_camera(c2[1], c2[2], W, H, cam2)
    p = subprocess.run([os.path.join(ROOT, "tests", "_build", "aruco_stereo_calibration"), str(raw1), str(raw2), str(W), str(H), str(len(f1)),
                        str(byml), "0.05", str(cam1), str(cam2), str(out)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    views, rms_cpp = p.stdout.split()
    w32 = lambda a: np.asarray(a, np.float32).astype(np.float64)
    py = stereoCalibrate(objs, i1, i2, w32(c1[1]), w32(c1[2]), w32(c2[1]), w32(c2[2]), (W, H), detector=md)
    assert int(views) == len(objs) and abs(float(rms_cpp) - py[0]) <= 1e-6 * py[0]
    fs = cv2.FileStorage(str(out), cv2.FILE_STORAGE_READ)
    for name, want in zip("RTEF", py[5:9]):
        got = fs.getNode(name).mat()
        assert got.dtype == np.float64 and np.array_equal(got.reshape(want.shape), want), name
    fs.release()
