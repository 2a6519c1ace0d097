"""Camera calibration from planar board views on the device: cv::calibrateCamera with flags 0 (fx, fy, cx, cy, k1, k2, p1, p2,
k3 free; skew and k4..k6 zero), for one camera or for a whole rig in one launch (ab_calibrate_cameras, kernel k_calibrate)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import ArucoError, ab_calib_camera, ab_calib_result, ab_stereo_pair, ab_stereo_result

_detectors = {}


def _context(device: int, detector):
    """The context a call runs on: the given MarkerDetector's, or one kept per device for these functions."""
    if detector is not None:
        return detector
    if device not in _detectors:
        from .detector import MarkerDetector
        _detectors[device] = MarkerDetector(device)
    return _detectors[device]


def _points(views, dim, what):
    out = []
    for v in views:
        a = np.asarray(v)
        if a.size % dim:
            raise ArucoError(_lib.AB_E_INVALID, "%s: every view needs N x %d coordinates" % (what, dim))
        out.append(np.ascontiguousarray(a.reshape(-1, dim), dtype=np.float32))
    return out


def calibrateCameras(cameras: Sequence, device: int = 0, detector=None) -> List[Optional[tuple]]:
    """cameras: [(objectPoints, imagePoints, imageSize)] with cv2.calibrateCamera's arguments per camera (object points on the
    z = 0 plane, f32 as cv2 uses them).  All cameras are calibrated in one launch.  Returns, per camera, cv2's
    (rms, K, D, rvecs, tvecs), or None for a degenerate camera (non-planar points, fewer than 2 views, a view with fewer
    than 4 points, or views that do not determine the focal lengths)."""
    det = _context(device, detector)
    recs = (ab_calib_camera * max(len(cameras), 1))()
    keep, n_views = [], []
    for c, (objs, imgs, size) in enumerate(cameras):
        objs, imgs = _points(objs, 3, "objectPoints"), _points(imgs, 2, "imagePoints")
        if len(objs) != len(imgs) or any(len(o) != len(i) for o, i in zip(objs, imgs)):
            raise ArucoError(_lib.AB_E_INVALID, "camera %d: objectPoints and imagePoints differ in shape" % c)
        n = np.array([len(o) for o in objs], np.int32)
        obj = np.ascontiguousarray(np.concatenate(objs) if objs else np.zeros((0, 3), np.float32))
        img = np.ascontiguousarray(np.concatenate(imgs) if imgs else np.zeros((0, 2), np.float32))
        keep.append((n, obj, img))
        recs[c] = ab_calib_camera(int(size[0]), int(size[1]), len(objs), n.ctypes.data, obj.ctypes.data, img.ctypes.data)
        n_views.append(len(objs))
    res = (ab_calib_result * max(len(cameras), 1))()
    total = sum(n_views)
    rv, tv = np.zeros((max(total, 1), 3)), np.zeros((max(total, 1), 3))
    det._check(det._lib.ab_calibrate_cameras(det._h, len(cameras), recs, res, rv.ctypes.data, tv.ctypes.data))
    out, v0 = [], 0
    for c, nv in enumerate(n_views):
        r = res[c]
        if r.status != 0:
            out.append(None)
        else:
            K = np.array(r.K, np.float64).reshape(3, 3)
            D = np.array(r.D, np.float64).reshape(1, 5)
            rvecs = tuple(rv[v0 + v].reshape(3, 1).copy() for v in range(nv))
            tvecs = tuple(tv[v0 + v].reshape(3, 1).copy() for v in range(nv))
            out.append((float(r.rms), K, D, rvecs, tvecs))
        v0 += nv
    return out


def calibrateCamera(objectPoints, imagePoints, imageSize, device: int = 0, detector=None):
    """cv2.calibrateCamera(objectPoints, imagePoints, imageSize, None, None) on the device: returns (rms, K, D, rvecs, tvecs)
    with cv2's shapes and dtypes.  Raises ArucoError(AB_E_INVALID) for degenerate input (see calibrateCameras)."""
    r = calibrateCameras([(objectPoints, imagePoints, imageSize)], device=device, detector=detector)[0]
    if r is None:
        raise ArucoError(_lib.AB_E_INVALID, "calibrateCamera: degenerate input (non-planar object points, fewer than 2 views, a view "
                                            "with fewer than 4 points, or views that do not determine the focal lengths)")
    return r


# ---- stereo calibration: cv2.stereoCalibrate with CALIB_FIX_INTRINSIC (ab_stereo_calibrate, kernel k_stereo_calibrate) ----------
CALIB_FIX_INTRINSIC = 256  # cv2.CALIB_FIX_INTRINSIC (the package does not import cv2)
_DEFAULT_CRITERIA = (3, 30, 1e-6)  # cv2's TermCriteria(COUNT + EPS, 30, 1e-6)


def _camera(K, D, what):
    K = np.asarray(K, np.float64)
    if K.size != 9:
        raise ArucoError(_lib.AB_E_INVALID, "%s: the camera matrix must be 3 x 3" % what)
    d = np.zeros(5) if D is None else np.asarray(D, np.float64).ravel()
    if d.size not in (0, 4, 5):
        raise ArucoError(_lib.AB_E_INVALID, "%s: distortion must have 4 or 5 coefficients (k1 k2 p1 p2 [k3])" % what)
    return K.ravel(), np.concatenate([d, np.zeros(5 - d.size)])


def stereoCalibratePairs(pairs: Sequence, criteria=_DEFAULT_CRITERIA, device: int = 0, detector=None) -> List[Optional[tuple]]:
    """pairs: [(objectPoints, imagePoints1, imagePoints2, cameraMatrix1, distCoeffs1, cameraMatrix2, distCoeffs2)] with
    cv2.stereoCalibrate's arguments per camera pair (object points on the z = 0 plane, f32 as cv2 uses them; distortion with 5
    or 4 coefficients, or None).  All pairs are calibrated in one launch with TermCriteria `criteria` (type, max_iter, eps);
    the type must be COUNT + EPS (3), cv2's default, and anything else raises ArucoError(AB_E_INVALID).
    Returns, per pair, cv2.stereoCalibrateExtended's (rms, K1, D1, K2, D2, R, T, E, F, rvecs, tvecs, perViewErrors) with the
    given intrinsics, or None for a degenerate pair (no view, a view with fewer than 4 or collinear points, points off the
    z = 0 plane, or a pose initialisation or result that is not finite)."""
    if int(criteria[0]) != 3:
        raise ArucoError(_lib.AB_E_INVALID, "stereoCalibrate: criteria type must be COUNT + EPS (3), got %d" % int(criteria[0]))
    det = _context(device, detector)
    max_iter, eps = int(criteria[1]), float(criteria[2])
    recs = (ab_stereo_pair * max(len(pairs), 1))()
    keep, n_views, cams = [], [], []
    for c, (objs, imgs1, imgs2, K1, D1, K2, D2) in enumerate(pairs):
        objs, imgs1, imgs2 = _points(objs, 3, "objectPoints"), _points(imgs1, 2, "imagePoints1"), _points(imgs2, 2, "imagePoints2")
        if not (len(objs) == len(imgs1) == len(imgs2)) or any(not (len(o) == len(a) == len(b)) for o, a, b in zip(objs, imgs1, imgs2)):
            raise ArucoError(_lib.AB_E_INVALID, "pair %d: objectPoints, imagePoints1 and imagePoints2 differ in shape" % c)
        k1, d1 = _camera(K1, D1, "pair %d camera 1" % c)
        k2, d2 = _camera(K2, D2, "pair %d camera 2" % c)
        n = np.array([len(o) for o in objs], np.int32)
        cat = lambda v, dim: np.ascontiguousarray(np.concatenate(v) if v else np.zeros((0, dim), np.float32))
        obj, i1, i2 = cat(objs, 3), cat(imgs1, 2), cat(imgs2, 2)
        keep.append((n, obj, i1, i2))
        recs[c] = ab_stereo_pair(0, 0, len(objs), n.ctypes.data, obj.ctypes.data, i1.ctypes.data, i2.ctypes.data, (C.c_double * 9)(*k1),
                                 (C.c_double * 5)(*d1), (C.c_double * 9)(*k2), (C.c_double * 5)(*d2))
        n_views.append(len(objs))
        cams.append((k1.reshape(3, 3).copy(), d1.reshape(1, 5).copy(), k2.reshape(3, 3).copy(), d2.reshape(1, 5).copy()))
    res = (ab_stereo_result * max(len(pairs), 1))()
    total = max(sum(n_views), 1)
    rv, tv, pve = np.zeros((total, 3)), np.zeros((total, 3)), np.zeros((total, 2))
    det._check(det._lib.ab_stereo_calibrate(det._h, len(pairs), recs, max_iter, eps, res, rv.ctypes.data, tv.ctypes.data, pve.ctypes.data))
    out, v0 = [], 0
    for c, nv in enumerate(n_views):
        r = res[c]
        if r.status != 0:
            out.append(None)
        else:
            m = lambda a: np.array(a, np.float64).reshape(3, 3)
            rvecs = tuple(rv[v0 + v].reshape(3, 1).copy() for v in range(nv))
            tvecs = tuple(tv[v0 + v].reshape(3, 1).copy() for v in range(nv))
            out.append((float(r.rms),) + cams[c] + (m(r.R), np.array(r.T, np.float64).reshape(3, 1), m(r.E), m(r.F), rvecs, tvecs,
                                                    pve[v0:v0 + nv].copy()))
        v0 += nv
    return out


def stereoCalibrateExtended(objectPoints, imagePoints1, imagePoints2, cameraMatrix1, distCoeffs1, cameraMatrix2, distCoeffs2, imageSize,
                            flags=CALIB_FIX_INTRINSIC, criteria=_DEFAULT_CRITERIA, device: int = 0, detector=None):
    """cv2.stereoCalibrateExtended(..., flags=CALIB_FIX_INTRINSIC) on the device: (rms, K1, D1, K2, D2, R, T, E, F, rvecs, tvecs,
    perViewErrors).  Only CALIB_FIX_INTRINSIC is supported; imageSize is accepted for cv2's signature (unused under that
    flag).  Raises ArucoError(AB_E_INVALID) for other flags and for degenerate input (see stereoCalibratePairs)."""
    if int(flags) != CALIB_FIX_INTRINSIC:
        raise ArucoError(_lib.AB_E_INVALID, "stereoCalibrate: only flags = CALIB_FIX_INTRINSIC (256) is supported, got %d" % int(flags))
    r = stereoCalibratePairs([(objectPoints, imagePoints1, imagePoints2, cameraMatrix1, distCoeffs1, cameraMatrix2, distCoeffs2)],
                             criteria=criteria, device=device, detector=detector)[0]
    if r is None:
        raise ArucoError(_lib.AB_E_INVALID, "stereoCalibrate: degenerate input (no view, a view with fewer than 4 or collinear points, "
                                            "object points off the z = 0 plane, or a pose that is not determined)")
    return r


def stereoCalibrate(objectPoints, imagePoints1, imagePoints2, cameraMatrix1, distCoeffs1, cameraMatrix2, distCoeffs2, imageSize,
                    flags=CALIB_FIX_INTRINSIC, criteria=_DEFAULT_CRITERIA, device: int = 0, detector=None):
    """cv2.stereoCalibrate(..., flags=CALIB_FIX_INTRINSIC) on the device: (rms, K1, D1, K2, D2, R, T, E, F)."""
    return stereoCalibrateExtended(objectPoints, imagePoints1, imagePoints2, cameraMatrix1, distCoeffs1, cameraMatrix2, distCoeffs2,
                                   imageSize, flags, criteria, device, detector)[:9]
