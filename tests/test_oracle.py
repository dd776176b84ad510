"""The numpy oracle vs outputs of the unmodified reference (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from oracle import linetr_oracle as orc
from linetr_b200 import synthetic as syn
from tests import helpers as H

TOL = 2e-5  # descriptors are unit-norm fp32; two fp32 CPU implementations agree to ~1e-6


@pytest.mark.parametrize("name", H.ENC_CASES)
def test_forward_matches_reference(name):
    npz, meta = H.golden()
    case = meta["cases"][name]
    data = H.case_inputs(case)
    H.assert_checksum(data, case["checksum"])
    got = orc.line_transformer_forward(H.weights_for(case["weights"]), data)
    assert got.shape == npz[name].shape
    assert np.abs(got - npz[name]).max() < TOL


@pytest.mark.parametrize("name", H.FULL_CASES)
def test_forward_matches_reference_full_size(name):
    """cfg[2] / cfg[3]-sized images with the stand-in checkpoint: the oracle against the committed reference output."""
    npz, meta = H.standin()
    case = meta["cases"][name]
    data = H.case_inputs(case)
    H.assert_checksum(data, case["checksum"])
    want, got = H.sampled(npz, name, orc.line_transformer_forward(H.standin_weights(), data))
    assert got.shape == want.shape
    assert np.abs(got - want).max() < TOL


def test_forward_batched():
    npz, meta = H.golden()
    case = meta["cases"]["enc_B2_L12_T21"]
    data = H.stack([syn.make_image_inputs(s, case["L"], case["T"], tuple(case["ntok"])) for s in case["seeds"]])
    H.assert_checksum(data, case["checksum"])
    got = orc.line_transformer_forward(H.weights_for(case["weights"]), data)
    assert np.abs(got - npz["enc_B2_L12_T21"]).max() < TOL


def test_pair_matches_reference():
    npz, meta = H.golden()
    case = meta["cases"]["pair_L32_27"]
    a, b, _ = syn.make_pair_inputs(case["seed"], case["L0"], case["T"], n_lines1=case["L1"],
                                   n_real_tokens=tuple(case["ntok"]))
    H.assert_checksum(a, case["checksum0"])
    H.assert_checksum(b, case["checksum1"])
    mat, dk, d0, d1 = orc.match_pair(H.weights_for(case["weights"]), a, b, case["thr"])
    assert np.abs(d0 - npz["pair_L32_27_d0"]).max() < TOL
    assert np.abs(d1 - npz["pair_L32_27_d1"]).max() < TOL
    assert np.abs(dk - npz["pair_L32_27_dist"]).max() < 1e-4
    assert np.array_equal(mat, npz["pair_L32_27_mat"])
    assert int(mat.sum()) == case["n_matches"]


def test_nn_matcher_bit_exact():
    npz, _ = H.golden()
    e0, e1, _ = syn.make_descriptor_pair(51, 64, 48)
    for mutual in (True, False):
        mat, dist = orc.nn_matcher(e0, e1, 0.8, mutual)
        assert mat.dtype == np.float64 and mat.shape == (1, 64, 48)
        assert np.array_equal(mat, npz[f"nn_64_48_mat_m{int(mutual)}"])
        assert np.abs(dist - npz["nn_64_48_dist"]).max() < 1e-6
    mat, _ = orc.nn_matcher(e0, e1, 0.05, True)
    assert np.array_equal(mat, npz["nn_64_48_mat_thr005"])


def test_distmat_ties_clip_threshold():
    npz, _ = H.golden()
    for mutual in (True, False):
        got = orc.nn_matcher_distmat(npz["distmat_ties_in"], 0.5, mutual)
        assert np.array_equal(got, npz[f"distmat_ties_mat_m{int(mutual)}"])


def test_distmat_empty():
    assert orc.nn_matcher_distmat(np.zeros((1, 0, 5), np.float32), 0.8).shape == (1, 0, 5)
    assert orc.nn_matcher_distmat(np.zeros((1, 4, 0), np.float32), 0.8).shape == (1, 4, 0)


def test_subline2keyline():
    npz, meta = H.golden()
    c = meta["cases"]["s2k"]

    def adj(ns):
        A = np.zeros((len(ns), sum(ns)), dtype=np.float32)
        s = 0
        for i, n in enumerate(ns):
            A[i, s:s + n] = 1.0 / n
            s += n
        return A
    f0, f1, _ = syn.make_descriptor_pair(c["seed"], sum(c["nsub0"]), sum(c["nsub1"]))
    dist = orc.get_dist_matrix(f0[None], f1[None])[0]
    assert np.abs(dist - npz["s2k_dist_sub"]).max() < 1e-6
    dk = orc.subline2keyline(dist, adj(c["nsub0"]), adj(c["nsub1"]))
    assert np.abs(dk - npz["s2k_dist_key"]).max() < 1e-6
    assert np.array_equal(orc.nn_matcher_distmat(dk, 0.8, True), npz["s2k_mat"])


def test_shipped_checkpoint():
    """The shipped checkpoint's magnitudes (its stand-in, tests/helpers.standin_weights) against the reference."""
    sd = H.standin_weights()
    npz, meta = H.standin()
    case = meta["cases"]["real_enc_L16_T21"]
    data = H.case_inputs(case)
    H.assert_checksum(data, case["checksum"])
    want, got = H.sampled(npz, "real_enc_L16_T21", orc.line_transformer_forward(sd, data))
    assert np.abs(got - want).max() < TOL
    case = meta["cases"]["real_pair_L128"]
    a, b, _ = syn.make_pair_inputs(case["seed"], case["L"], case["T"])
    H.assert_checksum(a, case["checksum0"])
    H.assert_checksum(b, case["checksum1"])
    mat, dk, d0, d1 = orc.match_pair(sd, a, b, case["thr"])
    for name, d in (("real_pair_L128_d0", d0), ("real_pair_L128_d1", d1)):
        want, got = H.sampled(npz, name, d)
        assert np.abs(got - want).max() < TOL
    assert np.array_equal(orc.match_indices(mat), npz["real_pair_L128_mat_idx"])
    assert int(mat.sum()) == case["n_matches"]


def test_torch_timing_port_matches_oracle_and_reference():
    """oracle/linetr_oracle_torch.py (the CPU baseline that bench.py times) gives the same
    answers as the numpy oracle and the committed reference outputs."""
    from oracle import linetr_oracle_torch as port
    npz, meta = H.golden()
    for name in ("enc_L16_T21", "enc_L37_T5_ragged", "enc_L9_T21_nd2"):
        case = meta["cases"][name]
        got = port.line_transformer_forward(port.prepare(H.weights_for(case["weights"])), H.case_inputs(case)).numpy()
        assert np.abs(got - npz[name]).max() < TOL
    case = meta["cases"]["pair_L32_27"]
    a, b, _ = syn.make_pair_inputs(case["seed"], case["L0"], case["T"], n_lines1=case["L1"],
                                   n_real_tokens=tuple(case["ntok"]))
    mat, dk, d0, _ = port.match_pair(port.prepare(H.weights_for(case["weights"])), a, b, case["thr"])
    assert np.array_equal(mat, npz["pair_L32_27_mat"]) and np.abs(d0 - npz["pair_L32_27_d0"]).max() < TOL
