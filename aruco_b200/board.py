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

    # ---- calibration from detected boards (the reference's utils/aruco_calibration) -----------------------------------------
    @staticmethod
    def stack_views(results, BConf: BoardConfiguration, markerSizeMeters: float = -1.0, min_markers: int = 4):
        """The calibration correspondences of the frames in `results` ((prob, Board, markers) per frame, as detect_batch and
        fetch return them) that matched at least min_markers markers, stacked as the board stage stacks them
        (board_select_stack): per matched marker in detection order its 4 configuration corners -- times metres per pixel
        (markerSizeMeters / |corner 0 - corner 1| of the first marker) for a PIX configuration with a marker size -- and its
        4 image corners.  Returns (objectPoints, imagePoints): lists of f32 (N, 3) / (N, 2) arrays."""
        objp = {}
        for i, corners in zip(BConf.ids, BConf.objPoints):
            objp.setdefault(int(i), corners)  # the first configuration entry with an id wins
        mpp = 1.0
        if BConf.mInfoType == BoardConfiguration.PIX and markerSizeMeters > 0:
            c = BConf.objPoints[0].astype(np.float32)
            d = (c[0] - c[1]).astype(np.float64)
            mpp = float(np.float32(markerSizeMeters)) / float(np.sqrt((d * d).sum()))
        objs, imgs = [], []
        for _, board, _ in results:
            ms = [m for m in board if int(m.id) in objp]
            if len(ms) < min_markers:
                continue
            objs.append(np.concatenate([(objp[int(m.id)].astype(np.float64) * mpp).astype(np.float32) for m in ms]))
            imgs.append(np.concatenate([np.asarray(m.corners, np.float32).reshape(4, 2) for m in ms]))
        return objs, imgs

    def calibrate(self, results, imageSize, min_markers: int = 4, raw: bool = False):
        """cv2.calibrateCamera on the device from the armed board's detections: `results` is the [(prob, Board, markers)] list
        of detect_batch / fetch.  Frames with fewer than min_markers matched markers are skipped (stack_views).  Returns
        (rms, K, D, rvecs, tvecs) over the kept frames; with raw=True ((rms, K, D, rvecs, tvecs), objectPoints, imagePoints),
        the f32 points the device used."""
        from .calib import calibrateCamera
        if self._bconf is None:
            raise ArucoError(_lib.AB_E_STATE, "BoardDetector.calibrate: setParams first")
        objs, imgs = self.stack_views(results, self._bconf, self._markerSize, min_markers)
        r = calibrateCamera(objs, imgs, imageSize, detector=self._mdetector)
        return (r, objs, imgs) if raw else r

    @staticmethod
    def stack_stereo_views(results1, results2, BConf: BoardConfiguration, markerSizeMeters: float = -1.0, min_markers: int = 4):
        """The stereo correspondences of two cameras' detections of the same frames (results1[f] and results2[f], as detect_batch
        and fetch return them): per frame the configuration markers matched by both cameras, in camera 1's detection order,
        stacked as stack_views stacks them (4 configuration corners each, times metres per pixel for a PIX configuration with a
        marker size, and the 4 image corners in each camera).  Frames with fewer than min_markers common markers are skipped.
        Returns (objectPoints, imagePoints1, imagePoints2): lists of f32 (N, 3) / (N, 2) / (N, 2) arrays."""
        if len(results1) != len(results2):
            raise ArucoError(_lib.AB_E_INVALID, "stack_stereo_views: the two cameras have %d and %d frames" % (len(results1), len(results2)))
        objs, imgs1, imgs2 = [], [], []
        for (p1, b1, m1), (p2, b2, m2) in zip(results1, results2):
            in2 = {}
            for m in b2:
                in2.setdefault(int(m.id), m)
            both = Board()
            other = Board()
            for m in b1:
                if int(m.id) in in2 and all(int(x.id) != int(m.id) for x in both):
                    both.append(m)
                    other.append(in2[int(m.id)])
            o, i1 = BoardDetector.stack_views([(p1, both, m1)], BConf, markerSizeMeters, min_markers)
            if not o:
                continue
            _, i2 = BoardDetector.stack_views([(p2, other, m2)], BConf, markerSizeMeters, min_markers)
            objs.append(o[0])
            imgs1.append(i1[0])
            imgs2.append(i2[0])
        return objs, imgs1, imgs2

    def stereoCalibrate(self, results1, results2, K1, D1, K2, D2, min_markers: int = 4, raw: bool = False,
                        criteria=(3, 30, 1e-6)):
        """cv2.stereoCalibrate (CALIB_FIX_INTRINSIC) on the device from the armed board's detections in two cameras' frames
        (stack_stereo_views).  Returns (rms, K1, D1, K2, D2, R, T, E, F); with raw=True (that tuple, objectPoints, imagePoints1,
        imagePoints2), the f32 points the device used."""
        from .calib import stereoCalibrate
        if self._bconf is None:
            raise ArucoError(_lib.AB_E_STATE, "BoardDetector.stereoCalibrate: setParams first")
        objs, i1, i2 = self.stack_stereo_views(results1, results2, self._bconf, self._markerSize, min_markers)
        r = stereoCalibrate(objs, i1, i2, K1, D1, K2, D2, None, criteria=criteria, detector=self._mdetector)
        return (r, objs, i1, i2) if raw else r
