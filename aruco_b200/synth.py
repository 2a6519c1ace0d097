"""Seeded synthetic frames for the benchmark/parity configs C3/C4/C5 (SURVEY.md 8(d)) and for batches of board views.

numpy only (no cv2): white canvas, gx x gy grid of markers, one random homography over the whole
canvas (4 % inset, +-3 % corner jitter), bilinear sampling with white fill, 3x3 Gaussian blur sigma 0.8,
contrast 0.8*I+20, additive Gaussian noise.  Marker bitmaps follow the reference generators' bit layout:
FiducidalMarkers::createMarkerImage (src/arucofidmarkers.cpp:214-229) and MarkerCode::getImg
(src/highlyreliablemarkers.cpp:234-256).  Input generator only -- not on the detection path.
"""
from __future__ import annotations

import numpy as np

_FID_WORDS = (0x10, 0x17, 0x09, 0x0E)


def fiducidal_bits(marker_id: int) -> np.ndarray:
    """7x7 cell matrix (1 = white) of marker `marker_id` (arucofidmarkers.cpp:220-229)."""
    assert 0 <= marker_id < 1024
    m = np.zeros((7, 7), np.uint8)
    for y in range(5):
        val = _FID_WORDS[(marker_id >> (2 * (4 - y))) & 3]
        for x in range(5):
            m[y + 1, x + 1] = (val >> (4 - x)) & 1
    return m


def hrm_bits(code: str, n: int) -> np.ndarray:
    """(n+2)x(n+2) cell matrix of an HRM code string (highlyreliablemarkers.cpp:234-256)."""
    m = np.zeros((n + 2, n + 2), np.uint8)
    m[1:-1, 1:-1] = np.array([c == "1" for c in code], np.uint8).reshape(n, n)
    return m


def _homography(src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    A = np.zeros((8, 8))
    b = np.zeros(8)
    for i in range(4):
        x, y = src[i]
        u, v = dst[i]
        A[i] = [x, y, 1, 0, 0, 0, -x * u, -y * u]
        A[i + 4] = [0, 0, 0, x, y, 1, -x * v, -y * v]
        b[i], b[i + 4] = u, v
    h = np.linalg.solve(A, b)
    return np.append(h, 1.0).reshape(3, 3)


def grid_for(n_markers: int):
    return {50: (10, 5), 100: (10, 10)}.get(n_markers, (int(np.ceil(np.sqrt(n_markers))),) * 2)


def render_frame(W: int, H: int, n_markers: int, seed: int, sigma: float = 2.0, marker_px: int | None = None,
                 hrm_codes=None, hrm_n: int = 0, flips: int = 0, clean: bool = False, as_float: bool = False):
    """Returns (grey u8 HxW, truth) with truth = {'ids': [...], 'corners': (n,4,2) f64 image coords}."""
    rng = np.random.default_rng(seed)
    gx, gy = grid_for(n_markers)
    if marker_px is None:
        # 4K: 7 cells x 27 px = 189 px sides, so that after the canvas homography (4 % inset, +-3 % jitter: the contour
        # shrinks to as little as 0.85x) every contour stays above the detector's minimum length 0.04*3840*4 = 614 px;
        # with the 175 px of round 1 about 5 % of the markers fell below it and were (correctly) rejected
        marker_px = 189 if W >= 3000 else (140 if W >= 1900 else int(0.09 * W))
    canvas = np.full((H, W), 255.0, np.float32)
    ins = 0.04
    x0, y0 = ins * W, ins * H
    cw, ch = (W - 2 * x0) / gx, (H - 2 * y0) / gy
    assert marker_px + 8 <= min(cw, ch), "markers do not fit the grid"
    if hrm_codes is None:
        ids = rng.choice(1024, size=gx * gy, replace=False)
        ncell = 7
    else:
        ids = rng.permutation(len(hrm_codes))[: gx * gy]
        ncell = hrm_n + 2
    cell = marker_px // ncell
    side = cell * ncell
    truth_ids, truth_c = [], []
    k = 0
    for j in range(gy):
        for i in range(gx):
            if k >= n_markers or k >= len(ids):
                break
            mid = int(ids[k])
            k += 1
            bits = fiducidal_bits(mid) if hrm_codes is None else hrm_bits(hrm_codes[mid], hrm_n).copy()
            if flips and hrm_codes is not None:
                inner = bits[1:-1, 1:-1]
                pos = rng.choice(hrm_n * hrm_n, size=flips, replace=False)
                inner.reshape(-1)[pos] ^= 1
            px = int(round(x0 + i * cw + (cw - side) / 2))
            py = int(round(y0 + j * ch + (ch - side) / 2))
            canvas[py:py + side, px:px + side] = np.kron(bits, np.ones((cell, cell), np.uint8)).astype(np.float32) * 255
            truth_ids.append(mid)
            truth_c.append([[px, py], [px + side - 1, py], [px + side - 1, py + side - 1], [px, py + side - 1]])
    src = np.array([[0, 0], [W - 1, 0], [W - 1, H - 1], [0, H - 1]], np.float64)
    base = np.array([[x0, y0], [W - 1 - x0, y0], [W - 1 - x0, H - 1 - y0], [x0, H - 1 - y0]], np.float64)
    jit = rng.uniform(-0.03, 0.03, size=(4, 2)) * np.array([W, H])
    dst = base + jit
    Hm = _homography(src, dst)
    Hi = np.linalg.inv(Hm)
    out = np.empty((H, W), np.float32)
    xs = np.arange(W, dtype=np.float64)
    band = 256
    for ys in range(0, H, band):
        ye = min(H, ys + band)
        yy = np.arange(ys, ye, dtype=np.float64)[:, None]
        den = Hi[2, 0] * xs[None, :] + Hi[2, 1] * yy + Hi[2, 2]
        sx = (Hi[0, 0] * xs[None, :] + Hi[0, 1] * yy + Hi[0, 2]) / den
        sy = (Hi[1, 0] * xs[None, :] + Hi[1, 1] * yy + Hi[1, 2]) / den
        fx, fy = np.floor(sx), np.floor(sy)
        ax, ay = (sx - fx).astype(np.float32), (sy - fy).astype(np.float32)
        ix, iy = fx.astype(np.int64), fy.astype(np.int64)
        inside = (ix >= 0) & (iy >= 0) & (ix < W - 1) & (iy < H - 1)
        ixc, iyc = np.clip(ix, 0, W - 2), np.clip(iy, 0, H - 2)
        v = (canvas[iyc, ixc] * (1 - ax) * (1 - ay) + canvas[iyc, ixc + 1] * ax * (1 - ay)
             + canvas[iyc + 1, ixc] * (1 - ax) * ay + canvas[iyc + 1, ixc + 1] * ax * ay)
        out[ys:ye] = np.where(inside, v, np.float32(255))
    g = np.exp(-1.0 / (2 * 0.8 * 0.8))
    k3 = np.array([g, 1.0, g], np.float32) / np.float32(1 + 2 * g)
    p = np.pad(out, 1, mode="edge")
    out = p[:, :-2] * k3[0] + p[:, 1:-1] * k3[1] + p[:, 2:] * k3[2]
    out = out[:-2] * k3[0] + out[1:-1] * k3[1] + out[2:] * k3[2]
    out = out * np.float32(0.8) + np.float32(20)
    if as_float:  # noise-free f32 image: the caller adds its own noise (bench: on the GPU, per frame)
        tc = np.array(truth_c, np.float64)
        ph = np.concatenate([tc, np.ones(tc.shape[:2] + (1,))], axis=2) @ Hm.T
        return out, {"ids": truth_ids, "corners": ph[..., :2] / ph[..., 2:3], "canvas_corners": tc}
    if not clean and sigma > 0:
        out = out + rng.normal(0.0, sigma, size=out.shape).astype(np.float32)
    grey = np.clip(np.rint(out), 0, 255).astype(np.uint8)
    tc = np.array(truth_c, np.float64)
    ph = np.concatenate([tc, np.ones(tc.shape[:2] + (1,))], axis=2) @ Hm.T
    tc_img = ph[..., :2] / ph[..., 2:3]
    return grey, {"ids": truth_ids, "corners": tc_img, "canvas_corners": tc}


def camera_for(W: int, H: int):
    """Synthetic pinhole camera of SURVEY 8(d): fx=fy=W, cx=W/2, cy=H/2, D=0."""
    K = np.array([[W, 0, W / 2], [0, W, H / 2], [0, 0, 1]], np.float32)
    D = np.zeros(5, np.float32)
    return K, D


def _board_frame_setup(board: np.ndarray, corners: np.ndarray):
    """The board's pixel -> centred-coordinate map, its outline and its marker corners in board image pixels."""
    bh, bw = board.shape
    ctr = np.array([[1, 0, -(bw // 2)], [0, 1, -(bh // 2)], [0, 0, 1]], np.float64)  # image pixel -> centred board coordinate
    outline = np.array([[0, 0], [bw - 1, 0], [bw - 1, bh - 1], [0, bh - 1]], np.float64)
    mk = np.asarray(corners, np.float64)[:, :, :2] + np.array([bw // 2, bh // 2], np.float64)
    return ctr, outline, mk


def _project(Hm, p):
    q = np.concatenate([p, np.ones(p.shape[:-1] + (1,))], axis=-1) @ Hm.T
    return q[..., :2] / q[..., 2:3]


def _draw_board_pose(rng, K, bh, W, H, max_tilt_deg):
    """One seeded board pose of warp_board: (R, t) in centred board-pixel units."""
    tilt, phi = np.radians(rng.uniform(0, max_tilt_deg)), rng.uniform(0, 2 * np.pi)
    psi = np.radians(rng.uniform(-20, 20))
    a = np.array([np.cos(phi), np.sin(phi), 0.0])  # in-plane tilt axis (Rodrigues)
    Ax = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    Rt = np.eye(3) + np.sin(tilt) * Ax + (1 - np.cos(tilt)) * Ax @ Ax
    Rz = np.array([[np.cos(psi), -np.sin(psi), 0], [np.sin(psi), np.cos(psi), 0], [0, 0, 1]])
    R = Rt @ Rz
    Z = K[0, 0] * bh / (rng.uniform(0.65, 0.8) * H)
    t = np.array([rng.uniform(-0.12, 0.12) * W * Z / K[0, 0], rng.uniform(-0.06, 0.06) * H * Z / K[0, 0], Z])
    return R, t


def _board_visible(Hm, outline, mk, W, H, min_chain, border):
    """warp_board's constraints: every board corner `border` inside the frame and every marker's 8-connected outline at least
    min_chain pixels."""
    o = _project(Hm, outline)
    if not ((o[:, 0] >= border * W).all() and (o[:, 0] <= (1 - border) * W).all() and (o[:, 1] >= border * H).all()
            and (o[:, 1] <= (1 - border) * H).all()):
        return False
    q = _project(Hm, mk)
    d = np.abs(q - np.roll(q, -1, axis=1))
    return np.max(d, axis=2).sum(axis=1).min() >= min_chain


def _render_board(board_f: np.ndarray, Hm: np.ndarray, W: int, H: int, rng, sigma: float) -> np.ndarray:
    """The board image (f32) under the homography Hm: bilinear sampling with white fill, render_frame's blur and additive
    Gaussian noise sigma drawn from rng.  Returns the u8 frame."""
    bh, bw = board_f.shape
    Hi = np.linalg.inv(Hm)
    xs = np.arange(W, dtype=np.float64)
    ys = np.arange(H, dtype=np.float64)[:, None]
    den = Hi[2, 0] * xs[None, :] + Hi[2, 1] * ys + Hi[2, 2]
    sx = (Hi[0, 0] * xs[None, :] + Hi[0, 1] * ys + Hi[0, 2]) / den
    sy = (Hi[1, 0] * xs[None, :] + Hi[1, 1] * ys + Hi[1, 2]) / den
    fx, fy = np.floor(sx), np.floor(sy)
    ax, ay = (sx - fx).astype(np.float32), (sy - fy).astype(np.float32)
    ix, iy = fx.astype(np.int64), fy.astype(np.int64)
    inside = (ix >= 0) & (iy >= 0) & (ix < bw - 1) & (iy < bh - 1)
    ixc, iyc = np.clip(ix, 0, bw - 2), np.clip(iy, 0, bh - 2)
    v = (board_f[iyc, ixc] * (1 - ax) * (1 - ay) + board_f[iyc, ixc + 1] * ax * (1 - ay)
         + board_f[iyc + 1, ixc] * (1 - ax) * ay + board_f[iyc + 1, ixc + 1] * ax * ay)
    img = np.where(inside, v, np.float32(255))
    # the 3x3 Gaussian (sigma 0.8) of render_frame: without it erosion breaks the thin threshold outlines of tilted edges
    g = np.exp(-1.0 / (2 * 0.8 * 0.8))
    k3 = np.array([g, 1.0, g], np.float32) / np.float32(1 + 2 * g)
    p = np.pad(img, 1, mode="edge")
    img = p[:, :-2] * k3[0] + p[:, 1:-1] * k3[1] + p[:, 2:] * k3[2]
    img = img[:-2] * k3[0] + img[1:-1] * k3[1] + img[2:] * k3[2]
    if sigma > 0:
        img = img + rng.normal(0.0, sigma, size=img.shape).astype(np.float32)
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def warp_board(board: np.ndarray, corners: np.ndarray, n_frames: int, W: int, H: int, seed: int, sigma: float = 1.5,
               max_tilt_deg: float = 40.0, min_chain: float = 240.0, border: float = 0.03):
    """n_frames views of a rendered board (u8 image, white background) through the pinhole camera of camera_for(W, H), each
    with its own seeded pose -- tilt of the board plane up to max_tilt_deg, in-plane rotation up to 20 degrees, the board
    filling 65-80 % of the frame height -- bilinear sampling with white fill, render_frame's blur and additive Gaussian
    noise sigma.  corners:
    the board configuration in pixels, centred on the image centre (createBoardImage), (n, 4, 3).  A pose is redrawn until
    every board corner lies `border` inside the frame and every marker's 8-connected outline (sum over its sides of
    max(|dx|, |dy|)) is at least min_chain pixels.  Returns (frames u8 [n_frames, H, W], homographies [n_frames, 3, 3] from
    board image pixels to frame pixels)."""
    rng = np.random.default_rng(seed)
    bh, bw = board.shape
    K, _ = camera_for(W, H)
    K = K.astype(np.float64)
    ctr, outline, mk = _board_frame_setup(board, corners)
    frames = np.empty((n_frames, H, W), np.uint8)
    homs = np.empty((n_frames, 3, 3))
    board_f = board.astype(np.float32)
    for f in range(n_frames):
        for _ in range(1000):
            R, t = _draw_board_pose(rng, K, bh, W, H, max_tilt_deg)
            Hm = K @ np.column_stack([R[:, 0], R[:, 1], t]) @ ctr
            if _board_visible(Hm, outline, mk, W, H, min_chain, border):
                break
        else:
            raise RuntimeError("warp_board: no pose satisfies the constraints")
        homs[f] = Hm
        frames[f] = _render_board(board_f, Hm, W, H, rng, sigma)
    return frames, homs


def warp_board_stereo(board: np.ndarray, corners: np.ndarray, n_frames: int, W: int, H: int, seed: int, R_lr, t_lr, sigma: float = 1.5,
                      max_tilt_deg: float = 40.0, min_chain: float = 240.0, border: float = 0.03):
    """n_frames pairs of views of a rendered board by two camera_for(W, H) cameras: camera 2 sees the camera-1 point x as
    R_lr x + t_lr (t_lr in the units of `corners`, board pixels).  Each frame draws one board pose as warp_board does (pose
    relative to camera 1) and redraws it until the board satisfies warp_board's border and outline constraints in both
    frames; both frames are rendered with warp_board's sampling, blur and noise.  Returns (frames1, frames2 u8 [n_frames, H,
    W], poses [n_frames, 3, 4]: camera 1's [R | t] of the board, in board pixels)."""
    rng = np.random.default_rng(seed)
    bh, bw = board.shape
    K, _ = camera_for(W, H)
    K = K.astype(np.float64)
    R_lr, t_lr = np.asarray(R_lr, np.float64).reshape(3, 3), np.asarray(t_lr, np.float64).reshape(3)
    ctr, outline, mk = _board_frame_setup(board, corners)
    frames1 = np.empty((n_frames, H, W), np.uint8)
    frames2 = np.empty((n_frames, H, W), np.uint8)
    poses = np.empty((n_frames, 3, 4))
    board_f = board.astype(np.float32)
    for f in range(n_frames):
        for _ in range(5000):
            R, t = _draw_board_pose(rng, K, bh, W, H, max_tilt_deg)
            R2, t2 = R_lr @ R, R_lr @ t + t_lr
            H1 = K @ np.column_stack([R[:, 0], R[:, 1], t]) @ ctr
            H2 = K @ np.column_stack([R2[:, 0], R2[:, 1], t2]) @ ctr
            if t2[2] > 0 and _board_visible(H1, outline, mk, W, H, min_chain, border) and _board_visible(H2, outline, mk, W, H, min_chain, border):
                break
        else:
            raise RuntimeError("warp_board_stereo: no pose satisfies the constraints in both frames")
        poses[f] = np.column_stack([R, t])
        frames1[f] = _render_board(board_f, H1, W, H, rng, sigma)
        frames2[f] = _render_board(board_f, H2, W, H, rng, sigma)
    return frames1, frames2, poses
