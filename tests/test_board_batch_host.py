"""The board stage's selection and stacking (board_select_stack, the AB_HD function k_board_batch runs per frame), compiled
for the host by tests/hostcheck/hostcheck_board.cpp, on the C++ oracle's markers of the golden board frames: the same
markers, object and image points as BoardDetector::detect on real OpenCV, and the pose solved from them agrees with
cv2.solvePnP."""
import ctypes as C

import numpy as np
import pytest

from conftest import ROOT, intrinsics, needs_cv2, rel_err

pytestmark = needs_cv2


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def hc(built):
    lib = C.CDLL(ROOT + "/tests/_build/libhostcheck.so")
    lib.hc_solve_pnp_planar.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p]
    sel = C.CDLL(ROOT + "/tests/_build/libhostcheck_board.so")
    sel.hc_board_select.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hc_board_select = sel.hc_board_select
    lib._board_lib = sel
    return lib


def mpp_of(cfg, size):
    """marker_meter_per_pix as the library computes it on the host: f32 corner differences, f64 norm."""
    if cfg["mInfoType"] != 0:
        return 1.0
    c = np.array(cfg["markers"][0]["corners"], np.float32)
    d = (c[0] - c[1]).astype(np.float64)
    return float(np.float64(np.float32(size))) / float(np.sqrt((d * d).sum()))


@pytest.mark.parametrize("name,cfgname,size", [("board", "board_pix", 1.0), ("chessboard", "chessboard_pix", 1.0),
                                               ("board", "board_meters", -1.0), ("chessboard", "chessboard_meters", -1.0)])
def test_board_select_matches_cv2_oracle(hc, frames, expected, name, cfgname, size):
    from aruco_b200._lib import ab_marker
    from oracle import cv2_oracle as o
    from oracle import native
    cfg = expected["boards"][cfgname]
    K, D = intrinsics(expected, name)
    ms = native.detect(frames[name], o.Params())["markers"]
    ms = ms + [{"id": 1023, "corners": np.zeros((4, 2), np.float32)}]  # an id outside the configuration is dropped
    buf = (ab_marker * len(ms))()
    for i, m in enumerate(ms):
        buf[i].id = int(m["id"])
        for j, v in enumerate(np.asarray(m["corners"], np.float32).reshape(8)):
            buf[i].corners[j] = float(v)
    ids = np.ascontiguousarray(np.array([m["id"] for m in cfg["markers"]], np.int32))
    cor = np.ascontiguousarray(np.array([m["corners"] for m in cfg["markers"]], np.float32).reshape(-1))
    n = len(ms)
    obj, img, slots = np.zeros((4 * n, 3), np.float32), np.zeros((4 * n, 2), np.float32), np.zeros(n, np.int32)
    nb = hc.hc_board_select(buf, n, P(ids), P(cor), len(ids), mpp_of(cfg, size), P(obj), P(img), P(slots))
    ref = o.board_detect(ms, cfg, K, D, size)
    assert [ms[s]["id"] for s in slots[:nb]] == [m["id"] for m in ref["markers"]] and nb == len(expected["goldens"][name]["markers"])
    # BoardDetector::detect's stacking as cv2_oracle.board_detect builds it (Point3f * double, detection order)
    pts = {m["id"]: np.array(m["corners"], np.float32) for m in cfg["markers"]}
    want_obj = np.array([(pts[m["id"]][p].astype(np.float64) * mpp_of(cfg, size)).astype(np.float32) for m in ref["markers"] for p in range(4)])
    want_img = np.array([np.asarray(m["corners"], np.float32)[p] for m in ref["markers"] for p in range(4)])
    assert np.array_equal(obj[:4 * nb].view(np.uint32), want_obj.view(np.uint32))
    assert np.array_equal(img[:4 * nb].view(np.uint32), want_img.view(np.uint32))
    r, t = np.zeros(3), np.zeros(3)
    o_, i_ = np.ascontiguousarray(obj[:4 * nb]), np.ascontiguousarray(img[:4 * nb])
    assert hc.hc_solve_pnp_planar(P(np.ascontiguousarray(K.ravel())), P(D), P(o_), P(i_), 4 * nb, P(r), P(t)) == 1
    assert rel_err(r, ref["rvec"]) < 1e-4 and rel_err(t, ref["tvec"]) < 1e-4
