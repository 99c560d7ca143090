"""`hot_counts`: poses_pnp's object availability count (pose_evaluation.py:183-190) restated in numpy on the LS
oracle's float32 softmax — the reference for casa_ls_vote_counts (tests/test_gpu_ls_device_eval.py).  Held here to the
golden vector of the reference's own poses_pnp (tests/golden/poses_pnp.npz), and at exact ties on the 0.1 boundary."""
import ast

import numpy as np

from oracle import golden_inputs as GI
from oracle import ls_voting_np as OL

from .test_golden_oracle import load


def hot_counts(seg, thresh=0.1):
    """Per image and class c >= 1 the pixels with softmax(seg * 1e6)[..., c] > thresh, compared in float32 (:183-188)
    -> [b, oc] int32."""
    hot = OL.hard_softmax_f32(np.asarray(seg, np.float32))[..., 1:]  # :183-185
    return (hot > np.float32(thresh)).sum(axis=(1, 2)).astype(np.int32)  # :186-188


def test_hot_counts_reproduce_the_golden_availability_mask():
    g = load("poses_pnp")
    gen = ast.literal_eval(str(g["gen"]))
    d, *_ = GI.pose_inputs(**gen)
    cnt = hot_counts(d["seg_logits"])
    b, oc = g["poses"].shape[:2]
    assert cnt.shape == (b, oc) and cnt.dtype == np.int32
    assert np.array_equal(cnt > 20, g["poses"].any(axis=(2, 3, 4)))


def test_hot_counts_at_exact_ties():
    """A k-way tie of the maximum gives hot = 1/k exactly: 1/10 rounds to 0.1f and is not counted, 1/9 is."""
    for k, counted in ((2, True), (3, True), (9, True), (10, False), (11, False)):
        seg = np.full((1, 1, 5, 12), -1.0, np.float32)
        seg[..., :k] = 0.5  # classes 0 .. k-1 tie (class 0, the background, is one of them)
        want = np.zeros(11, np.int32)
        want[:k - 1] = 5 if counted else 0
        assert np.array_equal(hot_counts(seg)[0], want), k
