"""Mirror of the caller of the hot path: aruco::BoardConfiguration / Board / BoardDetector
(src/board.h:56-140, src/boarddetector.{h,cpp}) -- SURVEY 8(f) "next" row 1.  The pose arithmetic (stacked
4*M-point planar solvePnP, reprojection-outlier re-solve, rotateXAxis) runs on the device: per call on given markers
(ab_detect_board), or for whole batches as one more kernel of the batch once setParams armed the board (ab_set_board)."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np

from . import _lib
from ._lib import ArucoError, ab_board, ab_board_config, ab_marker
from .detector import Marker, MarkerDetector


class BoardConfiguration:
    PIX, METERS = 0, 1

    def __init__(self, ids=(), objPoints=(), mInfoType=0):
        self.ids = [int(i) for i in ids]
        self.objPoints = np.asarray(objPoints, np.float32).reshape(-1, 4, 3)
        self.mInfoType = int(mInfoType)

    @staticmethod
    def from_dict(d) -> "BoardConfiguration":
        """d: {'mInfoType': 0|1, 'markers': [{'id': .., 'corners': 4x3}, ...]} (the aruco_bc_* YAML layout)."""
        return BoardConfiguration([m["id"] for m in d["markers"]], [m["corners"] for m in d["markers"]], d["mInfoType"])

    def size(self):
        return len(self.ids)

    def getMarkerInfo(self, marker_id):  # src/board.cpp:60-66
        for i, k in enumerate(self.ids):
            if k == marker_id:
                return self.objPoints[i]
        raise ArucoError(_lib.AB_E_INVALID, "Marker with the id given is not found")


class Board(list):
    """vector<Marker> + conf + Rvec/Tvec (src/board.h:103-140)."""

    def __init__(self):
        super().__init__()
        self.conf: Optional[BoardConfiguration] = None
        self.Rvec = None
        self.Tvec = None


class BoardDetector:
    def __init__(self, setYPerpendicular: bool = False, device: int = 0, detector: Optional[MarkerDetector] = None):
        self._setYPerpendicular = bool(setYPerpendicular)
        self.repj_err_thres = -1.0  # boarddetector.cpp:38-41
        self._mdetector = detector or MarkerDetector(device)
        self._bconf: Optional[BoardConfiguration] = None
        self._cam = (None, None)
        self._markerSize = -1.0
        self._vmarkers: List[Marker] = []
        self._boardDetected = Board()

    def setParams(self, bc: BoardConfiguration, camMatrix=None, distCoeff=None, markerSizeMeters: float = -1.0):
        """Also arms the board on the marker detector's context: its later batches (detect_batch, enqueue_device) run
        BoardDetector::detect on every frame.  bc None disarms."""
        self._bconf, self._cam, self._markerSize = bc, (camMatrix, distCoeff), float(markerSizeMeters)
        self._arm()

    def setYPerpendicular(self, enable: bool):
        self._setYPerpendicular = bool(enable)
        if self._bconf is not None:
            self._arm()

    def set_repj_err_thres(self, v: float):
        self.repj_err_thres = float(v)
        if self._bconf is not None:
            self._arm()

    def _arm(self):
        det = self._mdetector
        if self._bconf is None:
            det._check(det._lib.ab_set_board(det._h, None, None, None, -1.0, -1.0, 0))
            return
        cfg, keep = self._abi_config(self._bconf)
        Kf, Df = MarkerDetector._cam(*self._cam)
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        det._check(det._lib.ab_set_board(det._h, C.byref(cfg), p(Kf), p(Df), self._markerSize, float(self.repj_err_thres),
                                         int(self._setYPerpendicular)))

    @staticmethod
    def _abi_config(BConf: BoardConfiguration):
        """ab_board_config over contiguous copies of the configuration (returned too: they must outlive the call)."""
        ids = np.ascontiguousarray(np.array(BConf.ids, np.int32))
        pts = np.ascontiguousarray(BConf.objPoints.astype(np.float32).reshape(-1))
        return ab_board_config(len(ids), BConf.mInfoType, ids.ctypes.data, pts.ctypes.data), (ids, pts)

    def getMarkerDetector(self) -> MarkerDetector:
        return self._mdetector

    def getDetectedBoard(self) -> Board:
        return self._boardDetected

    def getDetectedMarkers(self) -> List[Marker]:
        return self._vmarkers

    def detect_image(self, image: np.ndarray) -> float:
        """BoardDetector::detect(const cv::Mat&) (boarddetector.cpp:66-78): markers first (no camera), then the board."""
        self._vmarkers = self._mdetector.detect(image)
        K, D = self._cam
        prob, self._boardDetected = self.detect(self._vmarkers, self._bconf, K, D, self._markerSize)
        return prob

    def detect(self, detectedMarkers: List[Marker], BConf: BoardConfiguration, camMatrix=None, distCoeff=None,
               markerSizeMeters: float = -1.0):
        """boarddetector.cpp:90-204. Returns (prob, Board)."""
        if BConf is None or BConf.size() == 0:
            raise ArucoError(_lib.AB_E_INVALID, "Invalid BoardConfig that is empty")  # CV_Assert (:93)
        det = self._mdetector
        n = len(detectedMarkers)
        buf = (ab_marker * max(n, 1))()
        for i, m in enumerate(detectedMarkers):
            buf[i].id = int(m.id)
            for j, v in enumerate(np.asarray(m.corners, np.float32).reshape(8)):
                buf[i].corners[j] = float(v)
            buf[i].ssize = float(m.ssize)
        cfg, keep = self._abi_config(BConf)
        Kf, Df = MarkerDetector._cam(camMatrix, distCoeff)
        outm = (ab_marker * max(n, 1))()
        res = ab_board()
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        det._check(det._lib.ab_detect_board(det._h, buf, n, C.byref(cfg), p(Kf), p(Df), float(markerSizeMeters),
                                            float(self.repj_err_thres), int(self._setYPerpendicular), outm, C.byref(res)))
        return float(res.prob), self._board(res, outm, 0, BConf)

    @staticmethod
    def _board(res, bm, off, BConf) -> Board:
        board = Board()
        board.conf = BConf
        for i in range(res.n_markers):
            m = bm[off + i]
            board.append(Marker(m.id, np.array(m.corners, np.float32).reshape(4, 2), m.ssize))
        if res.has_pose:
            board.Rvec = np.array(res.rvec, np.float64)
            board.Tvec = np.array(res.tvec, np.float64)
        return board

    # ---- batch path: the board stage runs inside the batch (setParams armed it) ---------------------------------------
    def _boards(self, markers: List[List[Marker]]):
        """(prob, Board, markers) per frame of the batch just returned by the marker detector."""
        det = self._mdetector
        n = len(markers)
        cap = max([1] + [len(m) for m in markers])
        res = (ab_board * max(n, 1))()
        bm = (ab_marker * (max(n, 1) * cap))()
        det._check(det._lib.ab_get_boards(det._h, n, res, bm, cap))
        return [(float(res[f].prob), self._board(res[f], bm, f * cap, self._bconf), markers[f]) for f in range(n)]

    def detect_batch(self, frames: np.ndarray):
        """BoardDetector::detect(const cv::Mat&) (boarddetector.cpp:66-78) over host frames [n,H,W] u8 or [n,H,W,3] BGR:
        markers without camera, then the armed board on each frame.  Returns [(prob, Board, markers)] per frame."""
        return self._boards(self._mdetector.detect_batch(frames))

    def enqueue_device(self, dev_ptr: int, width: int, height: int, n_frames: int, row_stride: Optional[int] = None,
                       frame_stride: Optional[int] = None):
        """Device-resident frames (two batches may be in flight, see MarkerDetector.enqueue_device); fetch returns them."""
        self._mdetector.enqueue_device(dev_ptr, width, height, n_frames, row_stride=row_stride, frame_stride=frame_stride)

    def fetch(self, n_frames: int, cap_per_frame: int = 256):
        """[(prob, Board, markers)] per frame of the oldest enqueued batch."""
        return self._boards(self._mdetector.fetch(n_frames, cap_per_frame))
