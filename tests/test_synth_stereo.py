"""synth.warp_board after its sampling was factored out for warp_board_stereo: byte-identical frames and homographies for the
seeds and frame counts the board-batch and calibration tests use (hashes of the implementation before the factoring), and
warp_board_stereo's constraints on both frames."""
import hashlib

import numpy as np

from aruco_b200 import synth

# sha256 of frames + homographies, from warp_board before _render_board / _draw_board_pose were factored out
WARP_BOARD_SHA256 = {(5, 30): "69b63573a235207a423ef1421011913f657db1772b1ada0dc5593ad1c92c985a",
                     (8, 64): "14a6c72eb3237630f77135d4e7cd9345ab425a34fc7517fb0431fe6cdfde741c"}


def _board():
    """A 4 x 6 marker board laid out as createBoardImage((4, 6), 100, 20) lays it out (100 px markers, 20 px gaps), drawn
    with numpy, and its centred pixel configuration."""
    rng = np.random.default_rng(0)
    img = np.full((740, 500), 255, np.uint8)
    corners = []
    for r in range(6):
        for c in range(4):
            x0, y0 = 20 + c * 120, 20 + r * 120
            img[y0:y0 + 100, x0:x0 + 100] = np.kron(synth.fiducidal_bits(int(rng.integers(1024))), np.ones((15, 15), np.uint8))[:100, :100] * 255
            corners.append([[x0 - 250, y0 - 370, 0], [x0 + 99 - 250, y0 - 370, 0], [x0 + 99 - 250, y0 + 99 - 370, 0], [x0 - 250, y0 + 99 - 370, 0]])
    return img, np.array(corners, np.float32)


def test_warp_board_frames_unchanged():
    img, cor = _board()
    for (seed, n), want in WARP_BOARD_SHA256.items():
        f, h = synth.warp_board(img, cor, n, 1280, 720, seed=seed)
        assert hashlib.sha256(f.tobytes() + h.tobytes()).hexdigest() == want, (seed, n)


def test_warp_board_stereo_keeps_the_board_inside_both_frames():
    img, cor = _board()
    W, H = 1280, 720
    R_lr = np.array([[np.cos(0.1), 0, np.sin(0.1)], [0, 1, 0], [-np.sin(0.1), 0, np.cos(0.1)]])
    t_lr = np.array([-180.0, 0, 0])
    f1, f2, poses = synth.warp_board_stereo(img, cor, 3, W, H, 7, R_lr, t_lr)
    assert f1.shape == f2.shape == (3, H, W) and f1.dtype == np.uint8 and poses.shape == (3, 3, 4)
    K = synth.camera_for(W, H)[0].astype(np.float64)
    outline = np.array([[-250, -370, 0], [249, -370, 0], [249, 369, 0], [-250, 369, 0]], np.float64)
    for f in range(3):
        R, t = poses[f][:, :3], poses[f][:, 3]
        for Rc, tc, frame in ((R, t, f1[f]), (R_lr @ R, R_lr @ t + t_lr, f2[f])):
            q = (K @ (outline @ Rc.T + tc).T).T
            q = q[:, :2] / q[:, 2:]
            assert (q[:, 0] >= 0.03 * W).all() and (q[:, 0] <= 0.97 * W).all() and (q[:, 1] >= 0.03 * H).all() and (q[:, 1] <= 0.97 * H).all()
            assert frame.min() < 60 and frame.max() > 200  # the board is drawn
