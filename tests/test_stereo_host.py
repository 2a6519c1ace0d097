"""Stereo calibration arithmetic (stereo_calibrate_t, ab_stereo.cuh -- what every CTA of k_stereo_calibrate runs), compiled for the
host by tests/hostcheck/hostcheck_stereo.cpp, against cv2.stereoCalibrateExtended (CALIB_FIX_INTRINSIC) on identical f32 inputs at
cv2's default and at converged criteria; cv2's output definitions checked as a black box; degenerate pairs; and
BoardDetector.stack_stereo_views against a numpy restatement."""
import numpy as np
import pytest

from conftest import needs_cv2
from stereo_data import CASES, CONVERGED, DEFAULT, case, compare, cv2_stereo, host_stereo

pytestmark = needs_cv2


@pytest.fixture(scope="module")
def hc(built):
    return True


def _args(d):
    return d["objs"], d["imgs1"], d["imgs2"], d["K1"], d["D1"], d["K2"], d["D2"]


@pytest.mark.parametrize("level", ["default", "converged"])
@pytest.mark.parametrize("c", CASES, ids=[str(c[0]) for c in CASES])
def test_host_stereo_matches_cv2(hc, c, level):
    d = case(c)
    crit = DEFAULT if level == "default" else CONVERGED
    st, got = host_stereo(*_args(d), criteria=crit)
    assert st == 0 and 1 <= got["iterations"] <= crit[1]
    compare(got, cv2_stereo(d, crit), d, level, "case %s" % (c,))


def test_cv2_output_definitions(hc):
    """The definitions the device reproduces, on cv2's own output: E = [T]x R, F = K2^-T E K1^-1 with F33 = 1, and rms and
    per-view errors from the same per-view sums (rms^2 = sum over views and cameras of n_v pve^2 / (2 sum n_v))."""
    d = case(CASES[0])
    r = cv2_stereo(d, CONVERGED)
    T = r["T"]
    Tx = np.array([[0, -T[2], T[1]], [T[2], 0, -T[0]], [-T[1], T[0], 0]])
    assert np.allclose(r["E"], Tx @ r["R"], rtol=0, atol=1e-12 * np.abs(r["E"]).max())
    F = np.linalg.inv(d["K2"]).T @ r["E"] @ np.linalg.inv(d["K1"])
    assert abs(r["F"][2, 2] - 1) < 1e-15 and np.allclose(r["F"], F / F[2, 2], rtol=1e-10, atol=0)
    n = np.array([len(o) for o in d["objs"]], np.float64)
    assert abs(np.sqrt((n[:, None] * r["pve"] ** 2).sum() / (2 * n.sum())) - r["rms"]) < 1e-12 * r["rms"]
    st, got = host_stereo(*_args(d), criteria=CONVERGED)
    assert abs(np.sqrt((n[:, None] * got["pve"] ** 2).sum() / (2 * n.sum())) - got["rms"]) < 1e-12 * got["rms"]


def _assert_degenerate(st, got):
    assert st == -1  # AB_E_INVALID
    for k in ("R", "T", "E", "F", "rvecs", "tvecs", "pve"):
        assert np.isfinite(got[k]).all() and not np.asarray(got[k]).any(), k
    assert got["rms"] == 0


def test_degenerate_pairs(hc):
    d = case(CASES[6])
    objs, i1, i2 = [list(x) for x in (d["objs"], d["imgs1"], d["imgs2"])]
    K = (d["K1"], d["D1"], d["K2"], d["D2"])
    _assert_degenerate(*host_stereo([], [], [], *K))
    three = [o.copy() for o in objs]
    _assert_degenerate(*host_stereo(three[:3] + [three[3][:3]], i1[:3] + [i1[3][:3]], i2[:3] + [i2[3][:3]], *K))
    bent = [o.copy() for o in objs]
    bent[0][:, 2] = np.linspace(0, 0.01, len(bent[0]), dtype=np.float32)
    _assert_degenerate(*host_stereo(bent, i1, i2, *K))
    _assert_degenerate(*host_stereo([o + np.float32([0, 0, 0.1]) for o in objs], i1, i2, *K))
    line = [o.copy() for o in objs]
    line[2][:, 1] = line[2][:, 0] * np.float32(0.5)  # every point of view 2 on one line
    _assert_degenerate(*host_stereo(line, i1, i2, *K))


# ---- BoardDetector.stack_stereo_views ------------------------------------------------------------------------------------------
def _restated(r1, r2, cfg, size, min_markers):
    pts = {}
    for i, c in zip(cfg.ids, cfg.objPoints):
        pts.setdefault(i, c)
    mpp = 1.0
    if cfg.mInfoType == 0 and size > 0:
        dd = (cfg.objPoints[0][0] - cfg.objPoints[0][1]).astype(np.float64)
        mpp = float(np.float32(size)) / float(np.sqrt((dd * dd).sum()))
    objs, a, b = [], [], []
    for (_, b1, _), (_, b2, _) in zip(r1, r2):
        c2 = {}
        for m in b2:
            c2.setdefault(m.id, m.corners)
        ids = []
        for m in b1:
            if m.id in pts and m.id in c2 and m.id not in ids:
                ids.append(m.id)
        if len(ids) < min_markers:
            continue
        c1 = {}
        for m in b1:
            c1.setdefault(m.id, m.corners)
        objs.append(np.concatenate([(pts[i].astype(np.float64) * mpp).astype(np.float32) for i in ids]))
        a.append(np.concatenate([np.asarray(c1[i], np.float32).reshape(4, 2) for i in ids]))
        b.append(np.concatenate([np.asarray(c2[i], np.float32).reshape(4, 2) for i in ids]))
    return objs, a, b


@pytest.mark.parametrize("size", [0.05, -1.0])
def test_stack_stereo_views_matches_numpy_restatement(size):
    from aruco_b200 import Board, BoardConfiguration, BoardDetector, Marker
    rng = np.random.default_rng(3)
    ids = list(range(10, 34))
    cfg = BoardConfiguration(ids, rng.uniform(-300, 300, (24, 4, 3)).astype(np.float32) * np.float32([1, 1, 0]), 0)

    def board(sel):
        b = Board()
        for i in sel:
            b.append(Marker(int(i), rng.uniform(0, 1000, (4, 2)).astype(np.float32)))
        return (len(b) / 24.0, b, list(b))
    frames1, frames2 = [], []
    for f in range(6):
        s1 = rng.permutation(ids + [99, 98])[: rng.integers(10, 26)]  # includes ids outside the configuration
        s2 = rng.permutation(ids)[: rng.integers(10, 25)]
        if f == 5:
            s1, s2 = ids[:3], ids[:3]  # below min_markers
        frames1.append(board(s1))
        frames2.append(board(s2))
    got = BoardDetector.stack_stereo_views(frames1, frames2, cfg, size, min_markers=4)
    want = _restated(frames1, frames2, cfg, size, 4)
    assert len(got[0]) == len(want[0]) >= 3
    for g, w in zip(got, want):
        for a, b in zip(g, w):
            assert a.dtype == np.float32 and np.array_equal(a.view(np.uint32), b.view(np.uint32))
