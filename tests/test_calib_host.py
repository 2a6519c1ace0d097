"""Camera calibration arithmetic (calibrate_camera_t, ab_calib.cuh -- what every CTA of k_calibrate runs), compiled for the host by
tests/hostcheck/hostcheck_calib.cpp, against cv2.calibrateCamera on identical f32 inputs; its degenerate-input reports; and
BoardDetector.stack_views (the points BoardDetector.calibrate hands to the device) against a numpy restatement on the golden
board frames."""
import numpy as np
import pytest

from calib_data import CASES, board_points, compare, cv2_calibrate, host_calibrate, make_views
from conftest import needs_cv2

pytestmark = needs_cv2


@pytest.fixture(scope="module")
def hc(built):
    return True


@pytest.mark.parametrize("seed,n_views,sigma,drop", CASES)
def test_host_calibration_matches_cv2(hc, seed, n_views, sigma, drop):
    W, H, objs, imgs = make_views(seed, n_views=n_views, sigma=sigma, drop=drop)
    st, got = host_calibrate(W, H, objs, imgs)
    assert st == 0
    assert 1 <= got["iterations"] <= 30
    compare(got, cv2_calibrate(W, H, objs, imgs), objs, "seed %d" % seed)


def _fronto_parallel(seed, sigma):
    import cv2
    rng = np.random.default_rng(seed)
    K = np.array([[1000.0, 0, 640], [0, 1000, 360], [0, 0, 1]])
    obj = board_points()
    objs, imgs = [], []
    for _ in range(10):
        rv = np.array([0, 0, rng.uniform(-1, 1)])
        tv = np.array([rng.uniform(-0.05, 0.05), rng.uniform(-0.03, 0.03), rng.uniform(0.4, 0.6)])
        p, _ = cv2.projectPoints(obj.astype(np.float64), rv, tv, K, np.zeros(5))
        objs.append(obj)
        imgs.append((p.reshape(-1, 2) + rng.normal(0, sigma, (len(obj), 2))).astype(np.float32))
    return 1280, 720, objs, imgs


def _assert_degenerate(st, got):
    assert st == -1  # AB_E_INVALID
    for k in ("K", "D", "rvecs", "tvecs"):
        assert np.isfinite(got[k]).all() and not got[k].any()
    assert got["rms"] == 0 and np.isfinite(got["rms"])


@pytest.mark.parametrize("seed,sigma", [(0, 0.0), (1, 0.0), (2, 0.0), (3, 0.01), (4, 0.01)])
def test_fronto_parallel_views_are_degenerate(hc, seed, sigma):
    """Every view parallel to the image plane: the focal length is not determined (cv2 returns f ~ 1e10)."""
    _assert_degenerate(*host_calibrate(*_fronto_parallel(seed, sigma)))


def test_non_planar_points_are_degenerate(hc):
    W, H, objs, imgs = make_views(3, n_views=10)
    objs = [o.copy() for o in objs]
    objs[0][:, 2] = np.linspace(0, 0.01, len(objs[0]), dtype=np.float32)
    _assert_degenerate(*host_calibrate(W, H, objs, imgs))
    # a plane at z = const != 0 is not the z = 0 plane cv::calibrateCamera requires
    W, H, objs, imgs = make_views(4, n_views=10)
    _assert_degenerate(*host_calibrate(W, H, [o + np.float32([0, 0, 0.1]) for o in objs], imgs))


def test_three_point_view_is_degenerate(hc):
    W, H, objs, imgs = make_views(5, n_views=10)
    objs, imgs = list(objs), list(imgs)
    objs[4], imgs[4] = objs[4][:3], imgs[4][:3]
    _assert_degenerate(*host_calibrate(W, H, objs, imgs))


@pytest.mark.parametrize("n", [0, 1])
def test_fewer_than_two_views_is_degenerate(hc, n):
    W, H, objs, imgs = make_views(6, n_views=3)
    _assert_degenerate(*host_calibrate(W, H, objs[:n], imgs[:n]))


# ---- BoardDetector.stack_views on the golden board frames ----------------------------------------------------------------
def _restated(frames_markers, cfg, size, min_markers):
    """numpy restatement of the board stage's stacking (board_select_stack): configuration corners times metres per pixel."""
    pts = {}
    for m in cfg["markers"]:
        pts.setdefault(m["id"], np.array(m["corners"], np.float32))
    mpp = 1.0
    if cfg["mInfoType"] == 0 and size > 0:
        c = np.array(cfg["markers"][0]["corners"], np.float32)
        d = (c[0] - c[1]).astype(np.float64)
        mpp = float(np.float32(size)) / float(np.sqrt((d * d).sum()))
    objs, imgs = [], []
    for ms in frames_markers:
        ms = [m for m in ms if m["id"] in pts]
        if len(ms) < min_markers:
            continue
        objs.append(np.array([(pts[m["id"]][p].astype(np.float64) * mpp).astype(np.float32) for m in ms for p in range(4)]))
        imgs.append(np.array([np.asarray(m["corners"], np.float32)[p] for m in ms for p in range(4)]))
    return objs, imgs


@pytest.mark.parametrize("name,cfgname,size", [("board", "board_pix", 0.05), ("chessboard", "chessboard_pix", 0.05),
                                               ("board", "board_meters", -1.0), ("board", "board_pix", -1.0)])
def test_stack_views_matches_numpy_restatement(frames, expected, name, cfgname, size):
    from aruco_b200 import Board, BoardConfiguration, BoardDetector, Marker
    from oracle import cv2_oracle as o
    from oracle import native
    cfg = expected["boards"][cfgname]
    bc = BoardConfiguration.from_dict(cfg)
    ms = native.detect(frames[name], o.Params())["markers"]
    # three "frames": all markers, all but the first three, and two markers (dropped by min_markers = 4)
    sets = [ms, ms[3:], ms[:2]]
    results = []
    for s in sets:
        b = Board()
        for m in s:
            if m["id"] in bc.ids:
                b.append(Marker(m["id"], np.asarray(m["corners"], np.float32).reshape(4, 2)))
        results.append((len(b) / bc.size(), b, s))
    objs, imgs = BoardDetector.stack_views(results, bc, size, min_markers=4)
    want_o, want_i = _restated([[m for m in s if m["id"] in bc.ids] for s in sets], cfg, size, 4)
    assert len(objs) == len(want_o) == 2
    for a, b, c, d in zip(objs, want_o, imgs, want_i):
        assert a.dtype == np.float32 and c.dtype == np.float32 and a.shape[1] == 3 and c.shape[1] == 2
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(c.view(np.uint32), d.view(np.uint32))
