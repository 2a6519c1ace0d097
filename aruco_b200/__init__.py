"""aruco_b200 -- B200-native implementation of ArUco's MarkerDetector::detect hot path.

Product code = aruco_b200/csrc (CUDA kernels + C ABI, built into aruco_b200/lib/libaruco_b200.so) and the
thin host mirror of the reference's operator interface in detector.py.  No CPU fallback exists.
"""
from .detector import FiducidalMarkers, HighlyReliableMarkers, Marker, MarkerDetector  # noqa: F401
from ._lib import ArucoError  # noqa: F401
from .board import Board, BoardConfiguration, BoardDetector  # noqa: F401
from .calib import calibrateCamera, calibrateCameras  # noqa: F401
from . import render  # noqa: F401

__all__ = ["MarkerDetector", "Marker", "FiducidalMarkers", "HighlyReliableMarkers", "ArucoError", "Board",
           "BoardConfiguration", "BoardDetector", "calibrateCamera", "calibrateCameras"]
