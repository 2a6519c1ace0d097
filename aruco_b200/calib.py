"""Camera calibration from planar board views on the device: cv::calibrateCamera with flags 0 (fx, fy, cx, cy, k1, k2, p1, p2,
k3 free; skew and k4..k6 zero), for one camera or for a whole rig in one launch (ab_calibrate_cameras, kernel k_calibrate)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import ArucoError, ab_calib_camera, ab_calib_result

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
