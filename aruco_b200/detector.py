"""Host-side mirror of the reference's operator interface for the hot path.

`MarkerDetector` has the names, argument meaning and error behaviour of aruco::MarkerDetector
(src/markerdetector.h:43-311 of the reference); `Marker` mirrors aruco::Marker (src/marker.h:46-141);
`FiducidalMarkers.detect` / `HighlyReliableMarkers.detect` are the two built-in decoders that can be passed
to setMakerDetectorFunction (markerdetector.h:243), recognised by identity and run on the device.  Every
method forwards to the C ABI (include/aruco_b200.h); nothing is computed in Python.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import ArucoError, ab_marker, ab_params


class Marker:
    """aruco::Marker: 4 corners (f32), id, ssize, Rvec/Tvec (f64, empty when no pose was computed)."""

    __slots__ = ("id", "corners", "ssize", "Rvec", "Tvec")

    def __init__(self, id=-1, corners=None, ssize=-1.0, Rvec=None, Tvec=None):
        self.id = id
        self.corners = np.zeros((4, 2), np.float32) if corners is None else np.asarray(corners, np.float32).reshape(4, 2)
        self.ssize = ssize
        self.Rvec = Rvec
        self.Tvec = Tvec

    def isValid(self):
        return self.id != -1 and self.corners.shape == (4, 2)

    def getCenter(self):  # src/marker.cpp:128-138
        return self.corners.astype(np.float32).sum(axis=0) / np.float32(4)

    def getPerimeter(self):
        d = self.corners - np.roll(self.corners, -1, axis=0)
        return float(np.sqrt((d.astype(np.float64) ** 2).sum(axis=1)).sum())

    def __lt__(self, other):  # src/marker.h:123
        return self.id < other.id

    def __repr__(self):
        return "Marker(id=%d, corners=%s)" % (self.id, self.corners.tolist())


class FiducidalMarkers:
    """Built-in decoder #1 (src/arucofidmarkers.h:90). `detect` is a sentinel: the device runs it."""

    @staticmethod
    def detect(canonical, n_rotations=None):
        raise RuntimeError("FiducidalMarkers.detect runs on the device inside MarkerDetector.detect")

    # generators (src/arucofidmarkers.h:49-88): drawn on the device, see aruco_b200/render.py
    @staticmethod
    def createMarkerImage(id, size, addWaterMark=False, locked=False):
        from . import render
        return render.createMarkerImage(id, size, addWaterMark, locked)

    @staticmethod
    def getMarkerMat(id):
        from . import render
        return render.getMarkerMat(id)

    @staticmethod
    def createBoardImage(gridSize, MarkerSize, MarkerDistance, ids):
        from . import render
        return render.createBoardImage(gridSize, MarkerSize, MarkerDistance, ids)

    @staticmethod
    def createBoardImage_ChessBoard(gridSize, MarkerSize, ids, centerData=True):
        from . import render
        return render.createBoardImage_ChessBoard(gridSize, MarkerSize, ids, centerData)

    @staticmethod
    def createBoardImage_Frame(gridSize, MarkerSize, MarkerDistance, ids, centerData=True):
        from . import render
        return render.createBoardImage_Frame(gridSize, MarkerSize, MarkerDistance, ids, centerData)


class HighlyReliableMarkers:
    """Built-in decoder #2 (src/highlyreliablemarkers.h:190-262). State is process-global like the reference's
    statics (highlyreliablemarkers.cpp:121-124); it is pushed to a detector when the decoder is selected."""

    _dict = None  # (n, bits uint8 [count, n*n], tau0, rate)

    @classmethod
    def loadDictionary(cls, dictionary, correctionDistanceRate: float = 1.0) -> bool:
        """dictionary: YAML text / path of a reference dictionary file, or (codes list[str], n, tau0)."""
        if isinstance(dictionary, str):
            text = dictionary
            if "\n" not in dictionary:
                with open(dictionary) as f:
                    text = f.read()
            kv = {}
            for line in text.splitlines():
                if ":" in line and not line.startswith("%"):
                    k, v = line.split(":", 1)
                    kv[k.strip()] = v.strip().strip('"')
            nm, n, tau0 = int(kv["nmarkers"]), int(kv["markersize"]), int(kv["tau0"])
            codes = [kv["marker_%d" % i] for i in range(nm)]
        else:
            codes, n, tau0 = dictionary
        if len(codes) == 0:
            return False
        bits = np.array([[c == "1" for c in s] for s in codes], np.uint8)
        cls._dict = (n, np.ascontiguousarray(bits), tau0, float(correctionDistanceRate))
        return True

    @staticmethod
    def detect(canonical, n_rotations=None):
        raise RuntimeError("HighlyReliableMarkers.detect runs on the device inside MarkerDetector.detect")


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class MarkerDetector:
    # enum ThresholdMethods (markerdetector.h:125) / CornerRefinementMethod (h:186)
    FIXED_THRES, ADPT_THRES, CANNY = 0, 1, 2
    NONE, HARRIS, SUBPIX, LINES = 0, 1, 2, 3

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.ab_create(device, C.byref(h))
        if rc != 0:
            raise ArucoError(rc, "ab_create failed (no CUDA device? this library has no CPU path)")
        self._h = h
        self._p = ab_params()
        self._lib.ab_default_params(C.byref(self._p))
        self._speed = 0
        self._cb_keep = None
        self._last_hw = None

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.ab_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ---- helpers -------------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise ArucoError(rc, self._lib.ab_last_error(self._h).decode())

    def _push(self):
        """Hands the edited parameter block to the library; a rejected value is rolled back (the local copy is
        refreshed from the library) so that it cannot poison later setters."""
        rc = self._lib.ab_set_params(self._h, C.byref(self._p))
        if rc != 0:
            msg = self._lib.ab_last_error(self._h).decode()
            self._lib.ab_get_params(self._h, C.byref(self._p))
            raise ArucoError(rc, msg)

    # ---- setters / getters (markerdetector.h:129-245) --------------------------------------------------
    def setThresholdMethod(self, m):
        self._p.thres_method = int(m)
        self._push()

    def getThresholdMethod(self):
        return self._p.thres_method

    def setThresholdParams(self, param1, param2):
        self._p.thres_param1, self._p.thres_param2 = float(param1), float(param2)
        self._push()

    def getThresholdParams(self):
        return self._p.thres_param1, self._p.thres_param2

    def setThresholdParamRange(self, r1=0, r2=0):  # markerdetector.h:152 (r2 is unused by the reference too)
        self._p.thres_param1_range = int(r1)
        self._push()

    def enableLockedCornersMethod(self, enable: bool):  # markerdetector.cpp:291-295
        self._p.locked_corners = int(bool(enable))
        if enable:
            self._p.corner_method = self.SUBPIX
        self._push()

    def enableErosion(self, enable: bool):  # API-compat extension (removed upstream, PortingManual.md:7)
        self._p.erosion = int(bool(enable))
        self._push()

    def setCornerRefinementMethod(self, m):
        self._p.corner_method = int(m)
        self._push()

    def getCornerRefinementMethod(self):
        return self._p.corner_method

    def setMinMaxSize(self, mn=0.03, mx=0.5):
        old = (self._p.min_size, self._p.max_size)
        self._p.min_size, self._p.max_size = float(mn), float(mx)
        try:
            self._push()
        except ArucoError:
            self._p.min_size, self._p.max_size = old
            raise

    def getMinMaxSize(self):
        return self._p.min_size, self._p.max_size

    def setDesiredSpeed(self, val):  # markerdetector.cpp:265-285 (val 3 falls through, SURVEY B.9)
        val = 0 if val < 0 else (2 if val > 3 else val)
        self._speed = val
        if val == 0:
            self._p.warp_size, self._p.corner_method = 56, self.SUBPIX
        elif val in (1, 2):
            self._p.warp_size, self._p.corner_method = 28, self.NONE
        self._push()

    def getDesiredSpeed(self):
        return self._speed

    def setWarpSize(self, val):
        old = self._p.warp_size
        self._p.warp_size = int(val)
        try:
            self._push()
        except ArucoError:
            self._p.warp_size = old
            raise

    def getWarpSize(self):
        return self._p.warp_size

    def setYPerpendicular(self, enable: bool):
        self._p.set_y_perpendicular = int(bool(enable))
        self._push()

    def setMakerDetectorFunction(self, fn):
        """Built-ins are recognised by identity and run on the device; any other callable
        fn(canonical: np.ndarray[S,S] uint8) -> (id, nRotations) is called back on the host."""
        if fn is FiducidalMarkers.detect or fn is FiducidalMarkers:
            self._p.decoder = 0
        elif fn is HighlyReliableMarkers.detect or fn is HighlyReliableMarkers:
            d = HighlyReliableMarkers._dict
            if d is None:
                raise ArucoError(_lib.AB_E_STATE, "HighlyReliableMarkers.loadDictionary must be called first")
            n, bits, tau0, rate = d
            self._check(self._lib.ab_load_hrm_dictionary(self._h, n, bits.shape[0], _ptr(bits), tau0, rate))
            self._p.decoder = 1
        else:
            def tramp(buf, size, nrot, _user):
                img = np.ctypeslib.as_array(buf, shape=(size, size))
                r = fn(img)
                mid, rot = (r if isinstance(r, tuple) else (r, 0))
                nrot[0] = int(rot)
                return int(mid)

            self._cb_keep = _lib.DECODER_FN(tramp)
            self._check(self._lib.ab_set_decoder_callback(self._h, self._cb_keep, None))
            self._p.decoder = 2
        self._push()

    def reserve(self, width, height, max_batch, max_quads=0, max_candidates=0, max_starts=0, max_points=0):
        self._check(self._lib.ab_reserve(self._h, width, height, max_batch, max_quads, max_candidates, max_starts, max_points))

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.ab_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    # ---- detect ---------------------------------------------------------------------------------------
    @staticmethod
    def _cam(K, D):
        Kf = None if K is None else np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        Df = None
        if D is not None:
            Df = np.zeros(5, np.float32)
            dd = np.asarray(D, np.float32).reshape(-1)[:5]
            Df[:len(dd)] = dd
        return Kf, Df

    def _markers(self, buf, counts, cap):
        out = []
        for f, n in enumerate(counts):
            ms = []
            for i in range(int(n)):
                m = buf[f * cap + i]
                mk = Marker(m.id, np.array(m.corners, np.float32).reshape(4, 2), m.ssize)
                if m.has_pose:
                    mk.Rvec = np.array(m.rvec, np.float64)
                    mk.Tvec = np.array(m.tvec, np.float64)
                ms.append(mk)
            out.append(ms)
        return out

    def detect_batch(self, frames: np.ndarray, camMatrix=None, distCoeff=None, markerSizeMeters: float = -1.0,
                     cap_per_frame: int = 256) -> List[List[Marker]]:
        """frames: uint8 [n, H, W] (grey) or [n, H, W, 3] (BGR, cvtColor front step)."""
        if frames.dtype != np.uint8 or frames.ndim not in (3, 4):
            raise ArucoError(_lib.AB_E_INVALID, "frames must be uint8 [n,H,W] or [n,H,W,3]")  # CV_Assert(8UC1), cpp:644
        frames = np.ascontiguousarray(frames)
        n, H, W = frames.shape[:3]
        Kf, Df = self._cam(camMatrix, distCoeff)
        buf = (ab_marker * (n * cap_per_frame))()
        counts = (C.c_int32 * n)()
        if frames.ndim == 3:
            rc = self._lib.ab_detect_batch(self._h, _ptr(frames), W, H, W, W * H, n, _ptr(Kf), _ptr(Df),
                                           float(markerSizeMeters), buf, cap_per_frame, counts)
        else:
            if frames.shape[3] != 3:
                raise ArucoError(_lib.AB_E_INVALID, "colour frames must be BGR (3 channels)")
            rc = self._lib.ab_detect_batch_bgr(self._h, _ptr(frames), W, H, 3 * W, 3 * W * H, n, _ptr(Kf), _ptr(Df),
                                               float(markerSizeMeters), buf, cap_per_frame, counts)
        self._check(rc)
        self._last_hw = (H, W)
        return self._markers(buf, list(counts), cap_per_frame)

    def detect(self, image: np.ndarray, camMatrix=None, distCoeff=None, markerSizeMeters: float = -1.0,
               setYPerpendicular: bool = False) -> List[Marker]:
        """MarkerDetector::detect (markerdetector.h:102): one frame, grey [H,W] or BGR [H,W,3]."""
        if bool(setYPerpendicular) != bool(self._p.set_y_perpendicular):
            self.setYPerpendicular(setYPerpendicular)
        return self.detect_batch(image[None], camMatrix, distCoeff, markerSizeMeters)[0]

    def enqueue_device(self, dev_ptr: int, width: int, height: int, n_frames: int, camMatrix=None, distCoeff=None,
                       markerSizeMeters: float = -1.0, row_stride: Optional[int] = None, frame_stride: Optional[int] = None):
        Kf, Df = self._cam(camMatrix, distCoeff)
        rs = width if row_stride is None else row_stride
        fs = rs * height if frame_stride is None else frame_stride
        self._check(self._lib.ab_enqueue_batch_device(self._h, C.c_void_p(dev_ptr), width, height, rs, fs, n_frames,
                                                      _ptr(Kf), _ptr(Df), float(markerSizeMeters)))
        self._last_hw = (height, width)

    def fetch(self, n_frames: int, cap_per_frame: int = 256, raw: bool = False):
        buf = (ab_marker * (n_frames * cap_per_frame))()
        counts = (C.c_int32 * n_frames)()
        self._check(self._lib.ab_fetch_results(self._h, buf, cap_per_frame, counts))
        if raw:
            return buf, list(counts)
        return self._markers(buf, list(counts), cap_per_frame)

    # ---- state of the last detect -----------------------------------------------------------------------
    def getThresholdedImage(self, frame: int = 0) -> np.ndarray:
        H, W = self._last_hw
        out = np.empty((H, W), np.uint8)
        self._check(self._lib.ab_get_thresholded(self._h, frame, _ptr(out), W))
        return out

    def getAllCandidates(self, frame: int = 0, cap: int = 1024):
        """Every candidate that reached the decoder: (quads [n,4,2], ids [n], nrot [n])."""
        q = np.zeros((cap, 4, 2), np.float32)
        ids = np.zeros(cap, np.int32)
        nr = np.zeros(cap, np.int32)
        n = C.c_int32()
        self._check(self._lib.ab_get_candidates(self._h, frame, _ptr(q), _ptr(ids), _ptr(nr), cap, C.byref(n)))
        return q[:n.value], ids[:n.value], nr[:n.value]

    def getCandidates(self, frame: int = 0):
        """MarkerDetector::getCandidates (h:266): the rejected quads."""
        q, ids, _ = self.getAllCandidates(frame)
        return q[ids < 0]

    def getCanonical(self, frame: int, candidate: int) -> np.ndarray:
        """S x S canonical image, S = the warp size the batch ran with (setWarpSize may have changed it since)."""
        S = C.c_int32()
        self._check(self._lib.ab_get_canonical_size(self._h, C.byref(S)))
        out = np.empty((S.value, S.value), np.uint8)
        self._check(self._lib.ab_get_canonical(self._h, frame, candidate, _ptr(out)))
        return out

    def getContour(self, frame: int, candidate: int, cap: int = 1 << 16) -> np.ndarray:
        xy = np.zeros((cap, 2), np.int32)
        n = C.c_int32()
        self._check(self._lib.ab_get_contour(self._h, frame, candidate, _ptr(xy), cap, C.byref(n)))
        return xy[:n.value]

    def counters(self):
        c = np.zeros(6, np.int64)
        self._check(self._lib.ab_get_counters(self._h, _ptr(c), 6))
        return dict(zip(("starts", "contours", "points", "quads", "candidates", "markers"), c.tolist()))

    def enable_timing(self, on=True):
        self._check(self._lib.ab_enable_timing(self._h, int(on)))

    def stage_ms(self):
        ms = np.zeros(5, np.float32)
        self._check(self._lib.ab_get_stage_ms(self._h, _ptr(ms), 5))
        return dict(zip(("threshold", "rectangles", "identify", "refine", "filter_pose"), ms.tolist()))

    KERNELS = ("threshold", "scan_starts", "trace", "trace_long", "emit", "polygon", "frame_filter", "sample", "identify", "refine", "finalize")

    def kernel_ms(self):
        ms = np.zeros(11, np.float32)
        self._check(self._lib.ab_get_kernel_ms(self._h, _ptr(ms), 11))
        return dict(zip(self.KERNELS, ms.tolist()))

    # ---- public workers (markerdetector.h:255-280) -----------------------------------------------------------
    def thresHold(self, method: int, grey: np.ndarray, param1: float = -1, param2: float = -1) -> np.ndarray:
        if grey.dtype != np.uint8 or grey.ndim != 2:
            raise ArucoError(_lib.AB_E_INVALID, "thresHold: grey must be 8UC1")  # CV_Assert, cpp:644
        grey = np.ascontiguousarray(grey)
        H, W = grey.shape
        out = np.empty_like(grey)
        self._check(self._lib.ab_threshold(self._h, _ptr(grey), W, H, W, int(method), float(param1), float(param2), _ptr(out), W))
        return out

    def detectRectangles(self, thres: np.ndarray, cap: int = 512) -> np.ndarray:
        thres = np.ascontiguousarray(thres)
        H, W = thres.shape
        q = np.zeros((cap, 4, 2), np.float32)
        n = C.c_int32()
        self._check(self._lib.ab_detect_rectangles(self._h, _ptr(thres), W, H, W, _ptr(q), cap, C.byref(n)))
        self._last_hw = (H, W)
        return q[:n.value]

    def warp(self, image: np.ndarray, size: int, points: Sequence) -> np.ndarray:
        pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1))
        if pts.size != 8:
            raise ArucoError(_lib.AB_E_INVALID, "warp: need 4 points")  # CV_Assert(points.size()==4), cpp:685
        image = np.ascontiguousarray(image)
        H, W = image.shape
        out = np.empty((size, size), np.uint8)
        self._check(self._lib.ab_warp(self._h, _ptr(image), W, H, W, _ptr(pts), int(size), _ptr(out)))
        return out

    def refineCandidateLines(self, corners, contour, camMatrix=None, distCoeff=None) -> np.ndarray:
        """MarkerDetector::refineCandidateLines (markerdetector.h:280, cpp:931-997): corners [4,2] (points of the
        contour), contour [n,2] int in the candidate's order -> refined corners [4,2] f32."""
        c = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(8)).copy()
        xy = np.ascontiguousarray(np.asarray(contour, np.int32).reshape(-1, 2))
        Kf, Df = self._cam(camMatrix, distCoeff)
        self._check(self._lib.ab_refine_candidate_lines(self._h, _ptr(xy), xy.shape[0], _ptr(c), _ptr(Kf), _ptr(Df)))
        return c.reshape(4, 2)

    def calculateExtrinsics(self, markers: List[Marker], markerSize: float, camMatrix, distCoeff=None,
                            setYPerpendicular: bool = False):
        """Marker::calculateExtrinsics (src/marker.cpp:112-125) for a list of markers (in place)."""
        n = len(markers)
        buf = (ab_marker * max(n, 1))()
        for i, m in enumerate(markers):
            buf[i].id = m.id
            for j, v in enumerate(np.asarray(m.corners, np.float32).reshape(8)):
                buf[i].corners[j] = float(v)
        Kf, Df = self._cam(camMatrix, distCoeff)
        self._check(self._lib.ab_calculate_extrinsics(self._h, buf, n, _ptr(Kf), _ptr(Df), float(markerSize), int(setYPerpendicular)))
        for i, m in enumerate(markers):
            m.Rvec = np.array(buf[i].rvec, np.float64)
            m.Tvec = np.array(buf[i].tvec, np.float64)
            m.ssize = float(markerSize)
        return markers
