"""-m gpu: BoardDetector over whole batches (ab_set_board / ab_get_boards, k_board_batch).  Every frame's board must be
byte-identical to ab_detect_board on that frame's fetched markers, and equal to the reference's goldens / cv2."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, have_cv2, intrinsics, rel_err

pytestmark = pytest.mark.gpu

CAP = 64
SYN_W, SYN_H, SYN_SIZE, SYN_SEED = 1280, 720, 0.05, 8


def P(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Armed:
    """A board configuration with the camera, as arrays the C ABI takes."""

    def __init__(self, cfg_dict, K, D, size, thr=-1.0, yperp=False):
        from aruco_b200._lib import ab_board_config
        self.d = cfg_dict
        self.ids = np.ascontiguousarray(np.array([m["id"] for m in cfg_dict["markers"]], np.int32))
        self.pts = np.ascontiguousarray(np.array([m["corners"] for m in cfg_dict["markers"]], np.float32).reshape(-1))
        self.cfg = ab_board_config(len(self.ids), cfg_dict["mInfoType"], self.ids.ctypes.data, self.pts.ctypes.data)
        self.K = None if K is None else np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
        self.D = None if D is None else np.ascontiguousarray(np.asarray(D, np.float32).reshape(5))
        self.size, self.thr, self.yperp = float(size), float(thr), int(yperp)

    def arm(self, det):
        assert det._lib.ab_set_board(det._h, C.byref(self.cfg), P(self.K), P(self.D), self.size, self.thr, self.yperp) == 0, \
            det._lib.ab_last_error(det._h)

    def config(self):
        from aruco_b200 import BoardConfiguration
        return BoardConfiguration.from_dict(self.d)


def disarm(det):
    assert det._lib.ab_set_board(det._h, None, None, None, -1.0, -1.0, 0) == 0


def detect_raw(det, frames):
    """ab_detect_batch without camera: the raw ab_marker buffer and the counts."""
    from aruco_b200._lib import ab_marker
    frames = np.ascontiguousarray(frames)
    n, H, W = frames.shape
    buf, cnt = (ab_marker * (n * CAP))(), (C.c_int32 * n)()
    det._check(det._lib.ab_detect_batch(det._h, P(frames), W, H, W, W * H, n, None, None, -1.0, buf, CAP, cnt))
    return buf, list(cnt)


def get_boards(det, n, cap=CAP):
    from aruco_b200._lib import ab_board, ab_marker
    res, bm = (ab_board * n)(), (ab_marker * (n * cap))()
    det._check(det._lib.ab_get_boards(det._h, n, res, bm, cap))
    return res, bm


def per_frame_board(det, a, buf, count, f):
    """ab_detect_board on frame f's fetched markers: (ab_board bytes, matched-marker bytes)."""
    from aruco_b200._lib import ab_board, ab_marker
    fm = (ab_marker * CAP).from_buffer(buf, f * CAP * C.sizeof(ab_marker))
    outm, res = (ab_marker * CAP)(), ab_board()
    det._check(det._lib.ab_detect_board(det._h, fm, count, C.byref(a.cfg), P(a.K), P(a.D), a.size, a.thr, a.yperp, outm, C.byref(res)))
    return bytes(res), bytes(outm)[:res.n_markers * C.sizeof(ab_marker)]


def assert_boards_equal_per_frame(det, a, buf, counts, res, bm, cap=CAP):
    from aruco_b200._lib import ab_marker
    ms = C.sizeof(ab_marker)
    for f in range(len(counts)):
        want_b, want_m = per_frame_board(det, a, buf, counts[f], f)
        assert bytes(res[f]) == want_b, f
        assert bytes(bm)[f * cap * ms:f * cap * ms + len(want_m)] == want_m, f


def paint_white(img, quads, grow=1.05):
    """the convex quads (4x2 corners), grown about their centres, filled white"""
    out = img.copy()
    yy, xx = np.mgrid[0:img.shape[0], 0:img.shape[1]]
    for q in quads:
        q = np.asarray(q, np.float64)
        c = q.mean(axis=0)
        q = c + (q - c) * grow
        d0, d1 = q[1] - q[0], q[2] - q[1]
        s = np.sign(d0[0] * d1[1] - d0[1] * d1[0])
        inside = np.ones(img.shape, bool)
        for k in range(4):
            p0, p1 = q[k], q[(k + 1) % 4]
            inside &= s * ((p1[0] - p0[0]) * (yy - p0[1]) - (p1[1] - p0[1]) * (xx - p0[0])) >= 0
        out[inside] = 255
    return out


def golden_batch(frames, expected, name):
    """the golden frame; 3 of its markers painted white; seeded noise; seeded small homography warps (cv2); `single`."""
    base = frames[name]
    g = expected["goldens"][name]["markers"]
    out = [base, paint_white(base, [m["corners"] for m in g[1:4]])]
    rng = np.random.default_rng(5)
    out.append(np.clip(base.astype(np.float64) + rng.normal(0, 3.0, base.shape), 0, 255).astype(np.uint8))
    if have_cv2():
        import cv2
        H, W = base.shape
        src = np.float32([[0, 0], [W - 1, 0], [W - 1, H - 1], [0, H - 1]])
        for _ in range(3):
            dst = (src + rng.uniform(-0.03, 0.03, (4, 2)) * np.float32([W, H])).astype(np.float32)
            out.append(cv2.warpPerspective(base, cv2.getPerspectiveTransform(src, dst), (W, H), borderValue=255))
    out.append(frames["single"])
    return np.ascontiguousarray(np.stack(out))


def check_api_and_cv2(bd, det, a, batch, buf, counts):
    """BoardDetector.detect_batch: every frame's Board equals BoardDetector.detect on that frame's markers, bit for bit;
    with cv2, the pose agrees with cv2_oracle.board_detect.  Returns the batch results."""
    bd.setParams(a.config(), None if a.K is None else a.K.reshape(3, 3), a.D, a.size)
    bd.set_repj_err_thres(a.thr)
    bd.setYPerpendicular(bool(a.yperp))
    out = bd.detect_batch(batch)
    assert len(out) == len(batch)
    o = None
    if have_cv2():
        from oracle import cv2_oracle as o
    for f, (prob, board, markers) in enumerate(out):
        assert len(markers) == counts[f]
        p1, b1 = bd.detect(markers, a.config(), None if a.K is None else a.K.reshape(3, 3), a.D, a.size)
        assert prob == p1 and [m.id for m in board] == [m.id for m in b1]
        assert all(np.array_equal(m.corners, m1.corners) and m.ssize == m1.ssize for m, m1 in zip(board, b1))
        assert (board.Rvec is None) == (b1.Rvec is None)
        if board.Rvec is not None:
            assert np.array_equal(board.Rvec, b1.Rvec) and np.array_equal(board.Tvec, b1.Tvec)
        if o is not None:
            ref = o.board_detect([{"id": m.id, "corners": m.corners} for m in markers], a.d, None if a.K is None else a.K.reshape(3, 3),
                                 a.D, a.size, a.thr, bool(a.yperp))
            assert [m["id"] for m in ref["markers"]] == [m.id for m in board]
            if board.Rvec is not None:
                assert rel_err(board.Rvec, ref["rvec"]) < 1e-4 and rel_err(board.Tvec, ref["tvec"]) < 1e-4
    return out


@pytest.fixture(scope="module")
def bd(built):
    from aruco_b200 import BoardDetector
    return BoardDetector()


@pytest.mark.parametrize("name", ["board", "chessboard"])
def test_goldens_through_the_batch(bd, frames, expected, name):
    det = bd.getMarkerDetector()
    K, D = intrinsics(expected, name)
    batch = golden_batch(frames, expected, name)
    cfgs = [(name + "_pix", 1.0, -1.0, False), (name + "_pix", 1.0, 1.5, False), (name + "_pix", 1.0, 0.8, True),
            (name + "_meters", -1.0, -1.0, False)]
    try:
        for cfgname, size, thr, yperp in cfgs:
            a = Armed(expected["boards"][cfgname], K, D, size, thr, yperp)
            a.arm(det)
            buf, counts = detect_raw(det, batch)
            res, bm = get_boards(det, len(batch))
            assert_boards_equal_per_frame(det, a, buf, counts, res, bm)
            out = check_api_and_cv2(bd, det, a, batch, buf, counts)
            if cfgname.endswith("_pix") and thr < 0:  # Aruco.Board / Aruco.Multi (test/core_tests.cpp:164-228) on frame 0
                g = expected["goldens"][name]
                prob, board, _ = out[0]
                assert [m.id for m in board] == [m["id"] for m in g["markers"]] and all(m.ssize == 1.0 for m in board)
                assert np.abs(board.Rvec - np.array(g["rvec"])).max() < 1e-4 and np.abs(board.Tvec - np.array(g["tvec"])).max() < 1e-4
                assert abs(prob - len(board) / len(a.ids)) < 1e-6
                painted = {m["id"] for m in g["markers"][1:4]}
                assert 0 < out[1][0] < prob and not painted & {m.id for m in out[1][1]}  # a partial board
        # no camera: the selection is still reported, probability 0, no pose (boarddetector.cpp:117-118)
        a = Armed(expected["boards"][name + "_pix"], None, None, 1.0)
        a.arm(det)
        buf, counts = detect_raw(det, batch)
        res, bm = get_boards(det, len(batch))
        assert_boards_equal_per_frame(det, a, buf, counts, res, bm)
        assert res[0].n_markers == len(expected["goldens"][name]["markers"]) and res[0].prob == 0.0 and res[0].has_pose == 0
        check_api_and_cv2(bd, det, a, batch, buf, counts)
    finally:
        bd.setParams(None)


@pytest.fixture(scope="module")
def synthetic(built, expected):
    """64 seeded views (tilt <= 40 deg, noise sigma 1.5) of a device-rendered 4x6 board (the ids of board_pix), 1280x720, and
    its configuration.  The seed is one whose views all keep their 24 markers after erosion."""
    from aruco_b200 import FiducidalMarkers, synth
    ids = [m["id"] for m in expected["boards"]["board_pix"]["markers"]]
    img, cfg = FiducidalMarkers.createBoardImage((4, 6), 100, 20, ids)
    batch, _ = synth.warp_board(img, cfg.objPoints, 64, SYN_W, SYN_H, seed=SYN_SEED)
    cfgd = {"mInfoType": cfg.mInfoType, "markers": [{"id": i, "corners": c.tolist()} for i, c in zip(cfg.ids, cfg.objPoints)]}
    return batch, cfgd


@pytest.fixture()
def c2det(built):
    """the C2 marker recipe: erosion + LINES, no camera"""
    from aruco_b200 import BoardDetector, MarkerDetector
    md = MarkerDetector(0)
    md.enableErosion(True)
    return BoardDetector(detector=md)


def synthetic_armed(cfgd):
    from aruco_b200 import synth
    K, D = synth.camera_for(SYN_W, SYN_H)
    return Armed(cfgd, K, D, SYN_SIZE)


def test_synthetic_multi_pose_batch(c2det, synthetic):
    batch, cfgd = synthetic
    det = c2det.getMarkerDetector()
    a = synthetic_armed(cfgd)
    a.arm(det)
    buf, counts = detect_raw(det, batch)
    assert counts == [24] * len(batch)
    res, bm = get_boards(det, len(batch))
    assert all(res[f].n_markers == 24 and res[f].has_pose and res[f].prob == 1.0 for f in range(len(batch)))
    assert_boards_equal_per_frame(det, a, buf, counts, res, bm)
    check_api_and_cv2(c2det, det, a, batch, buf, counts)


def test_pipeline_two_in_flight_and_host_chunks(c2det, synthetic):
    import torch
    batch, cfgd = synthetic
    det = c2det.getMarkerDetector()
    a = synthetic_armed(cfgd)
    a.arm(det)
    halves = (batch[:32], batch[32:])
    one = []  # one at a time
    for h in halves:
        buf, counts = detect_raw(det, h)
        one.append((bytes(buf), counts, get_boards(det, len(h))))
    dev = torch.from_numpy(batch).cuda()
    torch.cuda.synchronize()
    fs = SYN_W * SYN_H
    for i in range(2):
        det.enqueue_device(dev.data_ptr() + i * 32 * fs, SYN_W, SYN_H, 32)
    for i in range(2):
        buf, counts = det.fetch(32, CAP, raw=True)
        assert bytes(buf) == one[i][0] and counts == one[i][1]
        res, bm = get_boards(det, 32)  # the batch just fetched
        assert bytes(res) == bytes(one[i][2][0]) and bytes(bm) == bytes(one[i][2][1])
    # 80 host frames in chunks of 32 alternate between the two in-flight slots: the boards of the device path
    many = np.ascontiguousarray(np.concatenate([batch, batch[:16]]))
    dev80 = torch.from_numpy(many).cuda()
    torch.cuda.synchronize()
    det.enqueue_device(dev80.data_ptr(), SYN_W, SYN_H, 80)
    dbuf, dcounts = det.fetch(80, CAP, raw=True)
    dres, dbm = get_boards(det, 80)
    det.reserve(SYN_W, SYN_H, 32)
    hbuf, hcounts = detect_raw(det, many)
    hres, hbm = get_boards(det, 80)
    assert hcounts == dcounts and bytes(hbuf) == bytes(dbuf)
    assert bytes(hres) == bytes(dres) and bytes(hbm) == bytes(dbm)
    assert bytes(hres)[:len(bytes(one[0][2][0]))] == bytes(one[0][2][0])
    # setThresholdParamRange(2): five threshold images per frame
    det.setThresholdParamRange(2)
    try:
        buf, counts = detect_raw(det, batch[:8])
        res, bm = get_boards(det, 8)
        assert_boards_equal_per_frame(det, a, buf, counts, res, bm)
        assert all(res[f].has_pose for f in range(8))
    finally:
        det.setThresholdParamRange(0)


def test_errors_and_disarmed_markers_unchanged(built, synthetic):
    import torch
    from aruco_b200 import MarkerDetector
    from aruco_b200._lib import AB_E_CAPACITY, AB_E_INVALID, AB_E_STATE, ab_board, ab_board_config, ab_marker
    batch, cfgd = synthetic
    det = MarkerDetector(0)
    lib, h = det._lib, det._h
    a = synthetic_armed(cfgd)
    assert lib.ab_set_board(h, C.byref(ab_board_config(0, 0, a.ids.ctypes.data, a.pts.ctypes.data)), P(a.K), None, 1.0, -1.0, 0) == AB_E_INVALID
    assert lib.ab_set_board(h, C.byref(ab_board_config(24, 0, None, a.pts.ctypes.data)), P(a.K), None, 1.0, -1.0, 0) == AB_E_INVALID
    big_ids, big_pts = np.arange(1025, dtype=np.int32), np.zeros(1025 * 12, np.float32)
    assert lib.ab_set_board(h, C.byref(ab_board_config(1025, 0, big_ids.ctypes.data, big_pts.ctypes.data)), P(a.K), None, 1.0, -1.0, 0) == AB_E_INVALID
    # a batch that ran disarmed has no boards
    never = detect_raw(det, batch[:4])
    assert lib.ab_get_boards(h, 4, (ab_board * 4)(), None, CAP) == AB_E_STATE
    dev = torch.from_numpy(np.ascontiguousarray(batch[:4])).cuda()
    torch.cuda.synchronize()
    det.enqueue_device(dev.data_ptr(), SYN_W, SYN_H, 4)
    assert lib.ab_set_board(h, C.byref(a.cfg), P(a.K), P(a.D), a.size, -1.0, 0) == AB_E_STATE  # a batch in flight
    det.fetch(4, CAP)
    a.arm(det)
    detect_raw(det, batch[:4])
    assert lib.ab_get_boards(h, 4, (ab_board * 4)(), (ab_marker * 4 * 23)(), 23) == AB_E_CAPACITY  # 24 matched markers per frame
    assert lib.ab_get_boards(h, 3, (ab_board * 3)(), None, 0) == AB_E_STATE  # the batch had 4 frames
    assert lib.ab_get_boards(h, 4, (ab_board * 4)(), None, 0) == 0
    disarm(det)
    det.enqueue_device(dev.data_ptr(), SYN_W, SYN_H, 4)
    buf, counts = det.fetch(4, CAP, raw=True)
    assert bytes(buf) == bytes(never[0]) and counts == never[1]
    assert lib.ab_get_boards(h, 4, (ab_board * 4)(), None, 0) == AB_E_STATE


def test_cpp_facade_board_batch(bd, frames, expected, tmp_path):
    """tests/cpp/aruco_board_batch (BoardDetector::detectBatch of the C++ facade) on the golden board frames: the boards it
    saves, read back by cv::FileStorage, equal the Python batch results."""
    if not have_cv2():
        pytest.skip("cv2 needed to read the YAML back")
    import cv2
    exe = os.path.join(ROOT, "tests", "_build", "aruco_board_batch")
    ydir = os.path.join(ROOT, "tests", "golden", "yaml")
    batch = golden_batch(frames, expected, "board")
    n, H, W = batch.shape
    raw = tmp_path / "frames.raw"
    batch.tofile(str(raw))
    r = subprocess.run([exe, str(raw), str(W), str(H), str(n), os.path.join(ydir, "board__board_pix.yml"),
                        os.path.join(ydir, "board__intrinsics.yml"), "1.0", str(tmp_path / "board_")], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    K, D = intrinsics(expected, "board")
    a = Armed(expected["boards"]["board_pix"], K, D, 1.0)
    try:
        bd.setParams(a.config(), K, D, 1.0)
        bd.set_repj_err_thres(-1.0)
        bd.setYPerpendicular(False)
        out = bd.detect_batch(batch)
    finally:
        bd.setParams(None)
    rows = [l.split() for l in r.stdout.strip().splitlines()]
    assert len(rows) == n
    for f, (prob, board, markers) in enumerate(out):
        assert int(rows[f][0]) == len(markers) and abs(float(rows[f][1]) - prob) < 1e-6 and int(rows[f][2]) == len(board)
        fs = cv2.FileStorage(str(tmp_path / ("board_%d.yml" % f)), cv2.FILE_STORAGE_READ)
        b = fs.getNode("Board")
        if board.Rvec is not None:
            assert np.array_equal(np.array([b.getNode("Rvec").at(k).real() for k in range(3)]), board.Rvec)
            assert np.array_equal(np.array([b.getNode("Tvec").at(k).real() for k in range(3)]), board.Tvec)
        ms = b.getNode("Markers")
        got_ids = [int(ms.at(i).getNode("id").real()) for i in range(ms.size())] if ms.isSeq() else []  # an empty list is no sequence
        assert got_ids == [m.id for m in board]
        for i, m in enumerate(board):
            c = ms.at(i).getNode("corners")
            got = np.array([[c.at(k).at(0).real(), c.at(k).at(1).real()] for k in range(4)], np.float32)
            assert np.array_equal(got, m.corners)
