"""The L2 + LAB matching mode of the oracle (use_L2andLAB = True) against the reference's own code
(tests/golden/lab_pieces_golden.npz, written by tests/golden/make_lab_golden.py), and tf.argmin's rules.

Stated tolerances:
* rgb_to_lab: the reference evaluates pow in float32 and its 3x3 matmuls in an unpinned order; the oracle rounds
  an fp64 pow once and sums left to right.  Each output channel is one row of fxfyfz_to_lab, so the bound is
  4 ulp of that row's largest term (116 fy for L, 500 max(fx, fy) for a, 200 max(fy, fz) for b).
* the L2 distance: the reference's sum_x_square is a float32 reduce_sum and its sum_y_square a sum of float32
  squares; the oracle rounds float64 sums once.  Bound: 4 ulp of max(sum_x_square, sum_y_square).
"""
import os

import numpy as np
import torch
import torch.nn.functional as F

from oracle import dsin_oracle as O

import lab_oracle as L

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "lab_pieces_golden.npz"))


def _ulp(a):
    return np.spacing(np.abs(a).astype(np.float32)).astype(np.float64)


def _assert_lab_close(got, want):
    """Within 4 ulp of the largest term of each channel's fxfyfz_to_lab row (module docstring)."""
    got, want = got.reshape(-1, 3).astype(np.float64), want.reshape(-1, 3).astype(np.float64)
    fy = (want[:, 0] + 16.0) / 116.0
    fx, fz = fy + want[:, 1] / 500.0, fy - want[:, 2] / 200.0
    terms = [116.0 * fy, 500.0 * np.maximum(fx, fy), 200.0 * np.maximum(fy, fz)]
    for c in range(3):
        assert np.all(np.abs(got[:, c] - want[:, c]) <= 4 * _ulp(terms[c])), c


def test_rgb_to_lab_matches_the_reference_within_4_ulp_of_the_largest_term():
    want = GOLD["lab_out"]
    _assert_lab_close(L.rgb_to_lab(torch.tensor(GOLD["lab_in"])).numpy(), want)
    # the inputs reach both branches of both piecewise functions (f's threshold (6/29)^3 is at L = 8)
    v = GOLD["lab_in"]
    assert (v < np.float32(0.04045)).any() and (v > np.float32(0.04045)).any() and (v == np.float32(0.04045)).any()
    assert (want[:, 0] < 8.0).any() and (want[:, 0] > 8.0).any()
    # white on raw 0..255 values: L ~ 9342, far outside the usual 0..100
    white = L.rgb_to_lab(torch.tensor([[255.0, 255.0, 255.0]]))[0]
    assert 9341.0 < float(white[0]) < 9343.0 and float(white[1]) == 0.0 and float(white[2]) == 0.0


def test_lab_images_of_the_l2_case_match_the_reference():
    _assert_lab_close(O.extract_patches(L.rgb_to_lab(torch.tensor(GOLD["l2_x"])), 20, 24).numpy(), GOLD["l2_q"])
    _assert_lab_close(L.rgb_to_lab(torch.tensor(GOLD["l2_y"])).numpy(), GOLD["l2_r"])


def test_l2_distance_matches_the_reference_algebra_within_4_ulp():
    q, r = torch.tensor(GOLD["l2_q"]), torch.tensor(GOLD["l2_r"])
    got = L.l2_distances(q, r).permute(1, 2, 0).numpy().astype(np.float64)  # (h, w, P) as the reference
    want = GOLD["l2_out"].astype(np.float64)
    sx2 = (GOLD["l2_q"].astype(np.float64).reshape(4, -1) ** 2).sum(1)
    r64 = r.double().permute(2, 0, 1)[None]
    sy2 = F.conv2d(r64 * r64, torch.ones(1, 3, 20, 24, dtype=torch.float64))[0, 0].numpy()
    scale = np.maximum(sx2[None, None, :], sy2[:, :, None])
    assert np.all(np.abs(got - want) <= 4 * _ulp(scale))


def test_argmin_takes_the_first_of_exact_ties():
    """A search image holding the patch twice: two exact zeros, the first index wins."""
    rng = np.random.default_rng(3)
    q = rng.uniform(0, 9000, size=(20, 24, 3)).astype(np.float32)
    r = np.concatenate([rng.uniform(0, 9000, size=(3, 24, 3)).astype(np.float32), q, q], 0)
    d = L.l2_distances(torch.tensor(q)[None], torch.tensor(r))[0, :, 0]
    assert float(d[3]) == 0.0 and float(d[23]) == 0.0
    idx, best = L.l2_scores(torch.tensor(q)[None], torch.tensor(r), None)
    assert int(idx[0]) == 3 and float(best[0]) == 0.0


def test_argmin_lets_a_negative_distance_win_over_zero():
    """fp32 cancellation of ~1e10 terms makes a tiny true distance come out negative (-4096 here): it competes like
    any other value and beats the exact 0 of an identical window."""
    rng = np.random.default_rng(1)
    q = rng.uniform(3000, 9000, size=(20, 24, 3)).astype(np.float32)
    r = np.concatenate([rng.uniform(3000, 9000, size=(5, 24, 3)), q, q + rng.uniform(-0.01, 0.01, size=q.shape)])
    r = r.astype(np.float32)
    d = L.l2_distances(torch.tensor(q)[None], torch.tensor(r))[0, :, 0]
    assert float(d[5]) == 0.0 and float(d[25]) < 0.0
    idx, best = L.l2_scores(torch.tensor(q)[None], torch.tensor(r), None)
    assert int(idx[0]) == 25 and float(best[0]) == float(d[25])
