"""-m gpu: the canonical-image sampler (k_sample, k_warp_single) against cv2.warpPerspective(INTER_NEAREST).

k_sample evaluates each source coordinate in f32 and trusts it only when it lies clearly away from a rounding boundary;
every other pixel is deferred to OpenCV's f64 sequence, through a per-warp list of DECODE_LIST entries or, once that is
full, on the spot.  Markers whose quad side is (S-1)*k/2 with k odd put every other sample row and column exactly on a
half pixel, so most of their pixels are deferred and the list overflows.  The frames below are built for that:
fiducidal markers scaled by nearest neighbour onto quads with integer corners (the outer contour's corners, so the
candidate quads are known exactly), with weak noise so that a sample that rounds the wrong way changes the pixel."""
import numpy as np
import pytest

from test_gpu_parity import P_, check_frame, configure

pytestmark = pytest.mark.gpu

DECODE_LIST = 1024           # k_decode.cuh: per-warp list of deferred pixels
TIE_W, TIE_H = 1920, 1080
BLACK, WHITE = 36, 212       # grey levels: sigma-2 noise never clips, edges stay ~176 levels strong
MARGIN, GAP = 64, 24         # away from the border filter (0.025 * W = 48 px) and from each other
TIE_MIN_SIZE = 0.01          # smallest tie quad (S = 57, side 28) has a 112-point contour > 0.01 * 4 * 1920 = 76.8


# ---- frame builder (numpy only) -------------------------------------------------------------------------------------
def tie_geometries(S):
    """(shape, side, shear) for warp size S.  For odd S the sides (S-1)*k/2, k in {1, 3, 5}, and the shear (S-1)/2 put
    the samples on exact half pixels; side S-1 gives integer samples.  For even S, S-1 is odd and integer corners can
    only come near the ties: the sides are rounded down."""
    half = (S - 1) // 2
    out = [("axis", S - 1, 0)]
    for k in (1, 3, 5):
        L = (S - 1) * k // 2
        out += [("axis", L, 0), ("diamond", L, 0), ("para", L, half)]
    return out


def _corners(shape, L, a):
    """Integer corners relative to the bounding box's top-left, clockwise in image coordinates."""
    if shape == "axis":
        return np.array([[0, 0], [L, 0], [L, L], [0, L]])
    if shape == "diamond":
        return np.array([[L, 0], [2 * L, L], [L, 2 * L], [0, L]])
    return np.array([[0, 0], [L, 0], [L + a, L], [a, L]])  # parallelogram: sides (L, 0) and (a, L)


def _paint(img, q, bits):
    """Nearest-neighbour marker `bits` (7x7, 1 = white) on the parallelogram q (integer corners, q0 + q2 = q1 + q3): a
    pixel centre at q0 + u (q1 - q0) + v (q3 - q0), 0 <= u, v <= 1 takes cell (floor(7v), floor(7u))."""
    x0, y0 = q.min(axis=0)
    x1, y1 = q.max(axis=0)
    ys, xs = np.mgrid[y0:y1 + 1, x0:x1 + 1].astype(np.float64)
    e1, e2 = (q[1] - q[0]).astype(np.float64), (q[3] - q[0]).astype(np.float64)
    det = e1[0] * e2[1] - e1[1] * e2[0]
    px, py = xs - q[0][0], ys - q[0][1]
    u = (px * e2[1] - py * e2[0]) / det
    v = (py * e1[0] - px * e1[1]) / det
    eps = 1e-9
    inside = (u >= -eps) & (u <= 1 + eps) & (v >= -eps) & (v <= 1 + eps)
    cu = np.clip(np.floor(u * 7), 0, 6).astype(int)
    cv = np.clip(np.floor(v * 7), 0, 6).astype(int)
    val = np.where(bits[cv, cu] != 0, WHITE, BLACK).astype(np.float32)
    sub = img[y0:y1 + 1, x0:x1 + 1]
    sub[inside] = val[inside]


def tie_frames(S, seed, sigma=2.0, W=TIE_W, H=TIE_H):
    """Frames holding every tie_geometries(S) marker once (shelf-packed, as many frames as it takes).
    Returns [(grey u8 [H, W], [quad int [4, 2] per marker])]."""
    from aruco_b200 import synth
    rng = np.random.default_rng(seed)
    items = sorted(tie_geometries(S), key=lambda g: -_corners(*g).max(axis=0)[1])
    frames, cur = [], None
    x = y = row_h = 0
    for shape, L, a in items:
        c = _corners(shape, L, a)
        w, h = c.max(axis=0) + 1
        assert w + 2 * MARGIN <= W and h + 2 * MARGIN <= H, "marker does not fit the frame"
        if cur is not None and x + w > W - MARGIN:
            x, y, row_h = MARGIN, y + row_h + GAP, 0
        if cur is None or y + h > H - MARGIN:
            cur = (np.full((H, W), WHITE, np.float32), [])
            frames.append(cur)
            x, y, row_h = MARGIN, MARGIN, 0
        q = c + np.array([x, y])
        _paint(cur[0], q, synth.fiducidal_bits(int(rng.integers(1024))))
        cur[1].append(q)
        x += w + GAP
        row_h = max(row_h, h)
    out = []
    for img, quads in frames:
        if sigma > 0:
            img = img + rng.normal(0.0, sigma, img.shape).astype(np.float32)
        out.append((np.clip(np.rint(img), 0, 255).astype(np.uint8), quads))
    return out


# ---- references --------------------------------------------------------------------------------------------------
def _dst(S):
    return np.array([[0, 0], [S - 1, 0], [S - 1, S - 1], [0, S - 1]], np.float32)


def cv2_canonical(grey, quad, S):
    """MarkerDetector::warp (markerdetector.cpp:684-697) in real OpenCV."""
    import cv2
    M = cv2.getPerspectiveTransform(np.ascontiguousarray(quad, np.float32).reshape(4, 2), _dst(S))
    return cv2.warpPerspective(grey, M, (S, S), flags=cv2.INTER_NEAREST)


def deferred_count(quad, S):
    """Pixels k_sample defers to the f64 sequence for this quad: its f32 filter restated in numpy (f32 inverse map, the
    corner bound g, the same fused products rounded once).  Diagnostic: within a few pixels of the kernel's count."""
    import cv2
    M = cv2.getPerspectiveTransform(np.ascontiguousarray(quad, np.float32).reshape(4, 2), _dst(S))
    Mf = np.linalg.inv(M).astype(np.float32).astype(np.float64).ravel()
    e = float(S - 1)
    mx = my = 0.0
    sgn = []
    for cx, cy in ((0, 0), (e, 0), (0, e), (e, e)):
        d = Mf[6] * cx + Mf[7] * cy + Mf[8]
        sgn.append(d > 0)
        mx = max(mx, (abs(Mf[0]) * cx + abs(Mf[1]) * cy + abs(Mf[2])) / abs(d))
        my = max(my, (abs(Mf[3]) * cx + abs(Mf[4]) * cy + abs(Mf[5])) / abs(d))
    if len(set(sgn)) != 1:
        return S * S
    gx, gy = 0.5 - (4e-6 * mx + 2e-4), 0.5 - (4e-6 * my + 2e-4)
    f32 = np.float32
    y, x = np.mgrid[0:S, 0:S].astype(np.float64)
    den = f32(Mf[6] * x + f32(Mf[7] * y + Mf[8]).astype(np.float64))
    iden = (f32(1) / den).astype(np.float64)
    fx = f32(f32(Mf[0] * x + f32(Mf[1] * y + Mf[2]).astype(np.float64)).astype(np.float64) * iden)
    fy = f32(f32(Mf[3] * x + f32(Mf[4] * y + Mf[5]).astype(np.float64)).astype(np.float64) * iden)
    unc = ~((np.abs(fx) < 32768) & (np.abs(fy) < 32768)) | ~(np.abs(fx - np.rint(fx)) < gx) | ~(np.abs(fy - np.rint(fy)) < gy)
    return int(unc.sum())


def assert_canonicals_equal_cv2(det, grey, S, frame=0):
    """Every candidate's canonical image, bit for bit, against cv2 on the detector's own quad.  Returns the quads."""
    q, ids, _ = det.getAllCandidates(frame)
    assert len(q) > 0
    for i in range(len(q)):
        got, ref = det.getCanonical(frame, i), cv2_canonical(grey, q[i], S)
        bad = np.argwhere(got != ref)
        assert len(bad) == 0, "S=%d candidate %d %s: %d canonical pixels differ from cv2, first (y, x) %s: %d vs %d" % (
            S, i, q[i].tolist(), len(bad), bad[0].tolist(), got[tuple(bad[0])], ref[tuple(bad[0])])
    return q


@pytest.fixture(scope="module")
def det(built):
    from aruco_b200 import MarkerDetector
    d = MarkerDetector(0)
    d.reserve(TIE_W, TIE_H, 1, max_candidates=1024)
    return d


# ---- 1. ties and the full deferral list -------------------------------------------------------------------------
@pytest.mark.parametrize("S", [57, 65, 111, 127, 56])
def test_half_pixel_ties_and_full_deferral_list(det, S):
    """Tie quads at warp size S: every canonical image equals cv2's, and ids, rotations and every other stage equal both
    oracles.  At odd S the frames must drive at least one candidate past the DECODE_LIST deferred pixels, i.e. through
    the list-full branch."""
    P = P_(warp_size=S, min_size=TIE_MIN_SIZE)
    configure(det, P)
    counts = []
    for f, (grey, quads) in enumerate(tie_frames(S, seed=100 + S)):
        ms = det.detect(grey)
        q = assert_canonicals_equal_cv2(det, grey, S)
        check_frame(det, grey, P, markers=ms)
        # every marker of the builder reached the decoder on its exact quad (any start corner / orientation)
        got = {tuple(sorted(map(tuple, c.astype(int).tolist()))) for c in q}
        for c in quads:
            assert tuple(sorted(map(tuple, c.tolist()))) in got, "S=%d frame %d: quad %s not a candidate" % (S, f, c.tolist())
        counts += [deferred_count(c, S) for c in q]
    print("S=%d: deferred pixels per candidate (of %d): max %d, %d candidates > %d" % (
        S, S * S, max(counts), sum(c > DECODE_LIST for c in counts), DECODE_LIST))
    if S % 2:
        assert max(counts) > DECODE_LIST, "no candidate reaches the list-full branch"


# ---- 2. the whole warp-size range -------------------------------------------------------------------------------
SWEEP = [10, 11, 13, 21, 27, 56, 100, 110, 111, 112, 127, 128]  # S > 110: k_identify needs > 48 KB of shared memory


@pytest.mark.parametrize("S", SWEEP)
def test_warp_size_sweep(det, frames, S):
    """The golden frames and a seeded 1080p frame at every legal warp-size regime: S*S not a multiple of 4 (byte writes),
    S > 64 (OpenCV's 64-column blocks), S > 110 (the large-shared-memory k_identify launch), 10 and 128 (the bounds)."""
    from aruco_b200 import synth
    P = P_(warp_size=S)
    configure(det, P)
    for name in ("single", "board", "chessboard"):
        check_frame(det, frames[name], P)
        assert_canonicals_equal_cv2(det, frames[name], S)
    g, _ = synth.render_frame(1920, 1080, 50, seed=300 + S, sigma=2.0)
    ms, _ = check_frame(det, g, P)
    assert_canonicals_equal_cv2(det, g, S)
    if S >= 56:
        assert len(ms) >= 45


@pytest.mark.parametrize("S", [10, 128])
@pytest.mark.parametrize("n", [4, 6, 8])
def test_hrm_at_the_warp_size_bounds(det, expected, n, S):
    """HRM dictionaries at S = 10 (one pixel per cell for 8x8) and S = 128."""
    from aruco_b200 import HighlyReliableMarkers, synth
    text = expected["dictionaries"]["d%dx%d_100" % (n, n)]
    HighlyReliableMarkers.loadDictionary(text)
    codes = [l.split('"')[1] for l in text.splitlines() if l.startswith("marker_")]
    g, truth = synth.render_frame(1920, 1080, 50, seed=400 + n, sigma=2.0, hrm_codes=codes, hrm_n=n)
    P = P_(p1=21, p2=7, warp_size=S, decoder=1)
    configure(det, P)
    try:
        ms, _ = check_frame(det, g, P, hrm_text=text)
        assert_canonicals_equal_cv2(det, g, S)
    finally:
        configure(det, P_())
    if S == 128:  # (at S = 10 one pixel per cell misreads some codes, as the reference does)
        assert set(m.id for m in ms) <= set(truth["ids"]) and len(ms) >= 35


# ---- 3. batches, two in flight, re-reservation for a larger warp size -----------------------------------------------
def _state(d, f):
    q, ids, nrot = d.getAllCandidates(f)
    return q, list(ids), list(nrot), [d.getCanonical(f, i) for i in range(len(q))]


def _assert_same(got_markers, got_state, ref_markers, ref_state, what):
    assert [m.id for m in got_markers] == [m.id for m in ref_markers], what
    assert all((a.corners == b.corners).all() for a, b in zip(got_markers, ref_markers)), what
    gq, gids, grot, gcan = got_state
    rq, rids, rrot, rcan = ref_state
    assert gq.shape == rq.shape and (gq == rq).all() and gids == rids and grot == rrot, what
    for i, (a, b) in enumerate(zip(gcan, rcan)):
        assert a.shape == b.shape and (a == b).all(), "%s: canonical image %d differs" % (what, i)


def test_batches_and_warp_size_changes_between_them(built):
    """Eight tie frames through detect_batch and through enqueue_device with two batches in flight, the warp size raised
    from 56 to 128 and lowered to 10 between batches: every frame's candidates, canonical images and markers equal its
    single-frame result.  Raising S re-reserves the canonical buffers of the context and of its second in-flight set."""
    import torch
    from aruco_b200 import MarkerDetector
    sizes = (57, 65, 111, 127)
    frames = np.stack([tie_frames(sizes[i % 4], seed=500 + i)[0][0] for i in range(8)])
    B = len(frames)

    def setup(d, S):
        configure(d, P_(warp_size=S, min_size=TIE_MIN_SIZE))

    one = MarkerDetector(0)
    one.reserve(TIE_W, TIE_H, 1, max_candidates=1024)
    ref = {}
    for S in (56, 128, 10):
        setup(one, S)
        for f in range(B):
            ms = one.detect(frames[f])
            ref[S, f] = (ms, _state(one, 0))
            assert ref[S, f][1][3][0].shape == (S, S)
            assert_canonicals_equal_cv2(one, frames[f], S)
    assert sum(len(ref[56, f][0]) for f in range(B)) >= 8 * 10

    host = MarkerDetector(0)
    host.reserve(TIE_W, TIE_H, B, max_candidates=1024)
    for S in (56, 128, 10):
        setup(host, S)
        res = host.detect_batch(frames)
        for f in range(B):
            _assert_same(res[f], _state(host, f), *ref[S, f], "detect_batch S=%d frame %d" % (S, f))

    dev = MarkerDetector(0)
    dev.reserve(TIE_W, TIE_H, B, max_candidates=1024)
    d_frames = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()
    # (first batch S, second batch S): the second always runs on the second buffer set while the first is in flight
    for S0, S1 in ((56, 56), (56, 128), (128, 10)):
        setup(dev, S0)
        dev.enqueue_device(d_frames.data_ptr(), TIE_W, TIE_H, B)
        setup(dev, S1)
        dev.enqueue_device(d_frames.data_ptr(), TIE_W, TIE_H, B)
        for S in (S0, S1):
            res = dev.fetch(B)
            for f in range(B):
                _assert_same(res[f], _state(dev, f), *ref[S, f], "enqueue (%d, %d) batch S=%d frame %d" % (S0, S1, S, f))
    del d_frames


# ---- 4. the public warp worker ---------------------------------------------------------------------------------
@pytest.mark.parametrize("S", sorted(set(SWEEP + [56, 57, 65, 111, 127])))
def test_public_warp_equals_cv2(det, S):
    """MarkerDetector.warp (k_warp_single) on the tie quads, in all four start corners and both orientations."""
    for grey, quads in tie_frames(S, seed=600 + S):
        for q in quads:
            for r in range(4):
                for c in (np.roll(q, r, axis=0), np.roll(q[::-1], r, axis=0)):
                    c = c.astype(np.float32)
                    got, want = det.warp(grey, S, c), cv2_canonical(grey, c, S)
                    assert (got == want).all(), "S=%d quad %s: %d pixels differ" % (S, c.tolist(), int((got != want).sum()))
