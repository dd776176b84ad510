"""cfg[0] of BASELINE.json: the reference's `Matching` plugin / match_line_pairs.py path.

Two layers:
  * (CPU) the oracle against what the UNMODIFIED reference `Matching` produced on the four bundled image
    pairs (tests/golden/plumbing_pairs.npz: real SuperPoint descriptors, real line geometry, key lines split
    into sublines) - pins the oracle on real data, not only on synthetic inputs.  The matcher runs on the
    descriptors the reference computed with the shipped checkpoint; the line transformer runs with the
    checkpoint's stand-in (tests/helpers.standin_weights) against the reference's outputs with it;
  * (GPU) the captured tokeniser dicts replayed through the real plugin (tests/test_gpu_parity.py::test_plumbing_*).
"""
import numpy as np
import pytest

from oracle import linetr_oracle as orc
from tests import helpers as H


@pytest.mark.parametrize("pair", [0, 1, 2, 3])
def test_oracle_reproduces_reference_matching_on_real_pairs(pair):
    npz, meta = H.plumbing()
    snpz, smeta = H.standin()
    sd = H.standin_weights()
    info = meta["pairs"][pair]
    a, want0 = H.plumbing_image(npz, f"p{pair}_0")
    b, want1 = H.plumbing_image(npz, f"p{pair}_1")
    assert a["sublines"].shape[1] == info["S0"] and a["klines"].shape[1] == info["K0"]
    d0 = orc.line_transformer_forward(sd, a)
    d1 = orc.line_transformer_forward(sd, b)
    for side, d in ((0, d0), (1, d1)):
        want, got = H.sampled(snpz, f"p{pair}_{side}_line_desc", d)
        assert np.abs(got - want).max() < 2e-5
    A0, A1 = a["mat_klines2sublines"][0], b["mat_klines2sublines"][0]
    s2k = lambda d, A0, A1: orc.subline2keyline(d, A0, A1)
    mat, dk = H.matching_line_branch(orc.get_dist_matrix, s2k, orc.nn_matcher_distmat, d0, d1, A0, A1, 0.8)
    rows = snpz[f"p{pair}_scores_l_rows"]
    assert np.abs(dk[0][rows] - snpz[f"p{pair}_scores_l"]).max() < 1e-5    # descriptors differ by < 2e-5
    dec = snpz[f"p{pair}_decisive"]
    assert np.array_equal(orc.match_indices(mat)[dec], snpz[f"p{pair}_matches_l"][dec])
    # matcher on the REFERENCE descriptors of the shipped checkpoint: identical decisions, distances to fp32 rounding
    mat, dk = H.matching_line_branch(orc.get_dist_matrix, s2k, orc.nn_matcher_distmat, want0, want1, A0, A1, 0.8)
    assert np.abs(dk[0] - npz[f"p{pair}_scores_l"]).max() < 1e-6
    assert np.array_equal(orc.match_indices(mat), npz[f"p{pair}_matches_l"])
    assert int(mat.sum()) == info["n_matches_l"]


def test_oracle_point_branch_on_real_superpoint_descriptors():
    npz, meta = H.plumbing()
    mat, _ = orc.nn_matcher(npz["p0_desc_pnt0"], npz["p0_desc_pnt1"], 0.7, True)
    assert np.array_equal(orc.match_indices(mat), npz["p0_matches_p"])
    assert int(mat.sum()) == meta["pairs"][0]["n_matches_p"]
