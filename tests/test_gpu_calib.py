"""ab_calibrate_cameras / aruco_b200.calibrateCamera(s) / BoardDetector.calibrate on the device (k_calibrate): equal to the host
build of the same arithmetic and to cv2.calibrateCamera on identical f32 inputs, independent of the cameras sharing a launch,
bit-identical from run to run, its error returns, and end to end from rendered board views through the C++ driver."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from calib_data import CASES, compare, cv2_calibrate, host_calibrate, make_views
from conftest import ROOT, needs_cv2

pytestmark = [pytest.mark.gpu, needs_cv2]


def as_dict(r):
    rms, K, D, rv, tv = r
    return {"rms": rms, "K": K, "D": D.ravel(), "rvecs": [x.ravel() for x in rv], "tvecs": [x.ravel() for x in tv]}


@pytest.fixture(scope="module")
def det(built):
    from aruco_b200 import MarkerDetector
    return MarkerDetector(0)


@pytest.fixture(scope="module")
def sets():
    return [make_views(seed, n_views=n, sigma=s, drop=d) for seed, n, s, d in CASES]


def test_device_matches_host_build_and_cv2(det, sets):
    from aruco_b200 import calibrateCameras
    res = calibrateCameras([(o, i, (W, H)) for W, H, o, i in sets], detector=det)
    worst = {}
    for (W, H, objs, imgs), r, case in zip(sets, res, CASES):
        assert r is not None, case
        rms, K, D, rv, tv = r
        assert K.shape == (3, 3) and K.dtype == np.float64 and D.shape == (1, 5) and D.dtype == np.float64
        assert len(rv) == len(objs) and rv[0].shape == (3, 1) and tv[0].shape == (3, 1) and isinstance(rms, float)
        st, hc = host_calibrate(W, H, objs, imgs)
        assert st == 0
        for ref, name in ((hc, "host build"), (cv2_calibrate(W, H, objs, imgs), "cv2")):
            m = compare(as_dict(r), ref, objs, "case %s vs %s" % (case, name))
            for k, v in m.items():
                worst[(name, k)] = max(worst.get((name, k), 0.0), v)
    print("calibration maxima:", {"%s %s" % k: "%.3g" % v for k, v in sorted(worst.items())})


def _bits(r):
    return None if r is None else (np.float64(r[0]).tobytes(), r[1].tobytes(), r[2].tobytes(), np.concatenate(r[3]).tobytes(),
                                   np.concatenate(r[4]).tobytes())


def test_launch_composition_and_repeat_are_bit_identical(det, sets):
    """1, 7 and 300 cameras in one call each give exactly what the same camera gives alone; repeated calls are bit-identical."""
    from aruco_b200 import calibrateCameras
    cams = [(o, i, (W, H)) for W, H, o, i in sets]
    alone = [_bits(calibrateCameras([c], detector=det)[0]) for c in cams]
    assert [_bits(r) for r in calibrateCameras(cams[:1], detector=det)] == alone[:1]
    assert [_bits(r) for r in calibrateCameras(cams[3:10], detector=det)] == alone[3:10]
    order = [(7 * k + 3) % len(cams) for k in range(300)]
    big = calibrateCameras([cams[j] for j in order], detector=det)
    assert [_bits(r) for r in big] == [alone[j] for j in order]
    assert [_bits(r) for r in calibrateCameras([cams[j] for j in order], detector=det)] == [alone[j] for j in order]


def test_degenerate_camera_does_not_fail_the_call(det, sets):
    from aruco_b200 import ArucoError, calibrateCamera, calibrateCameras
    W, H, objs, imgs = sets[0]
    bad = [o.copy() for o in objs]
    bad[0][:, 2] = np.linspace(0, 0.01, len(bad[0]), dtype=np.float32)
    res = calibrateCameras([(objs, imgs, (W, H)), (bad, imgs, (W, H)), (objs[:1], imgs[:1], (W, H)),
                            ([objs[0], objs[1][:3]], [imgs[0], imgs[1][:3]], (W, H)), (objs, imgs, (W, H))], detector=det)
    assert res[1] is None and res[2] is None and res[3] is None
    assert _bits(res[0]) == _bits(res[4]) == _bits(calibrateCameras([(objs, imgs, (W, H))], detector=det)[0])
    with pytest.raises(ArucoError):
        calibrateCamera(bad, imgs, (W, H), detector=det)


def test_error_returns(det, sets):
    from aruco_b200 import _lib
    from aruco_b200._lib import ab_calib_camera, ab_calib_result
    lib, h = det._lib, det._h
    W, H, objs, imgs = sets[0]
    n = np.array([len(o) for o in objs], np.int32)
    obj, img = np.ascontiguousarray(np.concatenate(objs)), np.ascontiguousarray(np.concatenate(imgs))
    cam = ab_calib_camera(W, H, len(objs), n.ctypes.data, obj.ctypes.data, img.ctypes.data)
    out = ab_calib_result()
    assert lib.ab_calibrate_cameras(h, 1, C.byref(cam), C.byref(out), None, None) == 0 and out.status == 0
    assert lib.ab_calibrate_cameras(h, 1, None, C.byref(out), None, None) == _lib.AB_E_INVALID
    assert lib.ab_calibrate_cameras(h, 1, C.byref(cam), None, None, None) == _lib.AB_E_INVALID
    assert lib.ab_calibrate_cameras(h, -1, C.byref(cam), C.byref(out), None, None) == _lib.AB_E_INVALID
    assert lib.ab_calibrate_cameras(h, 65537, C.byref(cam), C.byref(out), None, None) == _lib.AB_E_INVALID
    assert b"65536" in lib.ab_last_error(h)
    for bad in (ab_calib_camera(W, H, -1, n.ctypes.data, obj.ctypes.data, img.ctypes.data),
                ab_calib_camera(W, H, 1025, n.ctypes.data, obj.ctypes.data, img.ctypes.data),
                ab_calib_camera(W, H, len(objs), None, obj.ctypes.data, img.ctypes.data),
                ab_calib_camera(W, H, len(objs), n.ctypes.data, None, img.ctypes.data),
                ab_calib_camera(W, H, len(objs), n.ctypes.data, obj.ctypes.data, None)):
        assert lib.ab_calibrate_cameras(h, 1, C.byref(bad), C.byref(out), None, None) == _lib.AB_E_INVALID
    big = np.array([4097], np.int32)
    cam2 = ab_calib_camera(W, H, 1, big.ctypes.data, obj.ctypes.data, img.ctypes.data)
    assert lib.ab_calibrate_cameras(h, 1, C.byref(cam2), C.byref(out), None, None) == _lib.AB_E_INVALID
    assert lib.ab_calibrate_cameras(h, 0, None, None, None, None) == 0


def test_state_error_while_a_batch_is_in_flight(built, sets):
    import torch
    from aruco_b200 import ArucoError, MarkerDetector, _lib, calibrateCamera
    from aruco_b200.synth import render_frame
    W, H, objs, imgs = sets[0]
    det = MarkerDetector(0)
    grey, _ = render_frame(640, 480, 4, seed=1)
    dev = torch.from_numpy(grey).cuda()
    torch.cuda.synchronize()
    det.enqueue_device(dev.data_ptr(), 640, 480, 1)
    with pytest.raises(ArucoError) as e:
        calibrateCamera(objs, imgs, (W, H), detector=det)
    assert e.value.code == _lib.AB_E_STATE
    det.fetch(1)
    ref = calibrateCamera(objs, imgs, (W, H))
    assert _bits(calibrateCamera(objs, imgs, (W, H), detector=det)) == _bits(ref)


# ---- end to end: rendered board views -> detect_batch -> calibrate, and the C++ driver ------------------------------------
@pytest.fixture(scope="module")
def board_views(built):
    from aruco_b200 import FiducidalMarkers
    from aruco_b200.synth import warp_board
    img, bc = FiducidalMarkers.createBoardImage((4, 6), 100, 20, list(range(24)))
    W, H = 1280, 720
    frames, _ = warp_board(img, bc.objPoints, 30, W, H, seed=5)
    return W, H, frames, bc


def test_end_to_end_from_rendered_views(board_views, tmp_path):
    from aruco_b200 import BoardDetector, MarkerDetector, calibrateCamera
    from aruco_b200.synth import camera_for
    W, H, frames, bc = board_views
    md = MarkerDetector(0)
    md.setCornerRefinementMethod(MarkerDetector.SUBPIX)  # as the C++ driver: LINES corners leave 0.7 px rms on these views
    bd = BoardDetector(detector=md)
    bd.setParams(bc, None, None, 0.05)
    results = bd.detect_batch(frames)
    (rms, K, D, rv, tv), objs, imgs = bd.calibrate(results, (W, H), raw=True)
    assert len(objs) >= 20 and all(o.dtype == np.float32 for o in objs) and all(i.dtype == np.float32 for i in imgs)
    got = {"rms": rms, "K": K, "D": D.ravel(), "rvecs": [x.ravel() for x in rv], "tvecs": [x.ravel() for x in tv]}
    print("end to end:", {k: v for k, v in compare(got, cv2_calibrate(W, H, objs, imgs), objs, "end to end").items()}, "rms %.4f" % rms)
    assert _bits((rms, K, D, rv, tv)) == _bits(calibrateCamera(objs, imgs, (W, H)))
    K0, _ = camera_for(W, H)
    assert abs(K[0, 0] / K0[0, 0] - 1) < 0.01 and abs(K[1, 1] / K0[1, 1] - 1) < 0.01
    assert abs(K[0, 2] - W / 2) < 0.02 * W / 2 and abs(K[1, 2] - H / 2) < 0.02 * H / 2
    # the C++ driver on the same frames writes intrinsics that readCameraParameters loads back
    raw = tmp_path / "frames.raw"
    raw.write_bytes(np.ascontiguousarray(frames).tobytes())
    byml, out = tmp_path / "board.yml", tmp_path / "intrinsics.yml"
    _save_board_config(bc, byml)
    p = subprocess.run([os.path.join(ROOT, "tests", "_build", "aruco_calibration"), str(raw), str(W), str(H), str(len(frames)), str(byml),
                        "0.05", str(out)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert abs(float(p.stdout.split()[-1]) - rms) <= 1e-6 * rms
    # readCameraParameters (through yaml_tool) loads K and D as the f32 values of the Python result
    yt = subprocess.run([os.path.join(ROOT, "tests", "_build", "yaml_tool"), "camera", str(out), str(tmp_path / "again.yml")],
                        capture_output=True, text=True, timeout=60)
    assert yt.returncode == 0, yt.stderr
    vals = yt.stdout.split()
    assert vals[0] == "camera" and (int(vals[1]), int(vals[2])) == (W, H)
    got_k = np.array(vals[3:12], np.float64).astype(np.float32)
    got_d = np.array(vals[12:17], np.float64).astype(np.float32)
    assert np.array_equal(got_k, K.astype(np.float32).ravel()) and np.array_equal(got_d, D.ravel().astype(np.float32))


def _save_board_config(bc, path):
    lines = ["%YAML:1.0", "---", "aruco_bc_nmarkers: %d" % bc.size(), "aruco_bc_mInfoType: %d" % bc.mInfoType, "aruco_bc_markers:"]
    for i, c in zip(bc.ids, bc.objPoints):
        pts = ", ".join("[ %r, %r, %r ]" % tuple(float(v) for v in p) for p in c)
        lines.append("   - { id:%d, corners:[ %s ] }" % (i, pts))
    path.write_text("\n".join(lines) + "\n")
