"""The C++ oracle's canonical images against cv2.warpPerspective(INTER_NEAREST) on the half-pixel tie frames of
test_gpu_sampler: the GPU tests compare k_sample with that oracle (check_frame), so it must itself equal OpenCV at the
inputs where rounding is decided by the last bit of the f64 source coordinate."""
import numpy as np
import pytest

from conftest import needs_cv2
from test_gpu_sampler import TIE_MIN_SIZE, cv2_canonical, deferred_count, tie_frames


@needs_cv2
@pytest.mark.parametrize("S", [57, 65, 111, 127, 56, 10, 128])
def test_oracle_canonical_equals_cv2_on_tie_frames(S):
    from oracle import native
    from oracle.cv2_oracle import Params
    for grey, quads in tie_frames(S, seed=100 + S):
        ref = native.detect(grey, Params(warp_size=S, min_size=TIE_MIN_SIZE), cap=2048)
        assert len(ref["quads"]) > 0
        for i, q in enumerate(ref["quads"]):
            want = cv2_canonical(grey, q, S)
            assert (ref["canon"][i] == want).all(), "S=%d candidate %d %s: %d pixels differ" % (
                S, i, q.tolist(), int((ref["canon"][i] != want).sum()))
        if S in (57, 65, 111, 127):  # every builder marker is a candidate, on its exact quad, and the ties are real
            got = {tuple(sorted(map(tuple, c.astype(int).tolist()))) for c in ref["quads"]}
            assert all(tuple(sorted(map(tuple, c.tolist()))) in got for c in quads)
            assert len(ref["markers"]) == len(quads)
            assert max(deferred_count(c, S) for c in ref["quads"]) > 1024
