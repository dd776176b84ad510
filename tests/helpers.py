"""Shared test helpers: golden fixtures, regenerated inputs, drift checks."""
import json
import os

import numpy as np

from linetr_b200 import synthetic as syn

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_cache = {}


def golden():
    if "npz" not in _cache:
        _cache["npz"] = dict(np.load(os.path.join(GOLDEN_DIR, "reference_outputs.npz")))
        with open(os.path.join(GOLDEN_DIR, "reference_outputs.json")) as f:
            _cache["meta"] = json.load(f)
    return _cache["npz"], _cache["meta"]


FULL_CASES = ["real_enc_L256_T32", "real_enc_L512_T64_ragged"]   # cases of standin()


def checksum(d):
    return {k: float(np.asarray(v, dtype=np.float64).sum()) for k, v in sorted(d.items())}


def assert_checksum(d, want):
    got = checksum(d)
    assert got.keys() == want.keys()
    for k in got:
        assert abs(got[k] - want[k]) <= 1e-6 * max(1.0, abs(want[k])), f"input generator drift in {k}"


def weights_for(tag):
    kind, *rest = tag.split(":")
    if kind == "synthetic":
        return syn.make_state_dict(int(rest[0]), int(rest[1]))
    if kind == "standin":
        return standin_weights()
    raise KeyError(tag)


STANDIN_SEED = 2024


def standin_weights():
    """Stand-in for the shipped LineTR checkpoint (22 MB, not part of the repository): every tensor is
    seeded normal noise with the mean and standard deviation of the shipped tensor, clipped to its range
    (golden/checkpoint_stats.json), so that BatchNorm statistics, LayerNorm gains and weight scales have
    the trained model's magnitudes.  golden/standin_outputs.npz holds what the reference computed with it."""
    if "standin" not in _cache:
        with open(os.path.join(GOLDEN_DIR, "checkpoint_stats.json")) as f:
            stats = json.load(f)
        rng = np.random.Generator(np.random.PCG64(STANDIN_SEED))
        sd = {}
        for key, shape, kind in syn.state_dict_spec(1):
            mean, std, lo, hi = stats[key]
            if kind == "bn_count":
                sd[key] = np.array(int(mean), dtype=np.int64)
            else:
                sd[key] = np.clip(mean + std * rng.standard_normal(shape), lo, hi).astype(np.float32)
        _cache["standin"] = sd
    return _cache["standin"]


def save_standin_checkpoint(path):
    """The stand-in as a checkpoint file (what LineTransformer(mode='test') loads)."""
    import torch
    torch.save({k: torch.from_numpy(v.copy()) for k, v in standin_weights().items()}, path)
    return str(path)


def standin():
    """Outputs of the reference with the stand-in checkpoint (tests/golden/make_standin_golden.py).  Large
    descriptor sets are stored as a seeded sample of lines: `<name>_cols` indexes the lines of `<name>`."""
    if "standin_npz" not in _cache:
        _cache["standin_npz"] = dict(np.load(os.path.join(GOLDEN_DIR, "standin_outputs.npz")))
        with open(os.path.join(GOLDEN_DIR, "standin_outputs.json")) as f:
            _cache["standin_meta"] = json.load(f)
    return _cache["standin_npz"], _cache["standin_meta"]


def sampled(npz, name, full):
    """(stored sample, the same lines of `full` [.., 256, L])."""
    cols = npz[f"{name}_cols"]
    return npz[name], full[..., cols]


def case_inputs(case):
    ntok = case.get("ntok")
    ntok = tuple(ntok) if isinstance(ntok, list) else ntok
    return syn.make_image_inputs(case["seed"], case["L"], case["T"], ntok)


def stack(images):
    return {k: np.concatenate([im[k] for im in images], axis=0) for k in images[0]}


ENC_CASES = ["enc_L16_T21", "enc_L1_T21", "enc_L37_T5_ragged", "enc_L24_T32_ragged", "enc_L130_T21",
             "enc_L9_T21_nd2"]


# ---------------------------------------------------------------- cfg[0] plumbing / tokenizer fixtures
TOK_KEYS = ("klines", "length_klines", "angles", "sublines", "pnt_sublines", "mask_sublines", "resp_sublines",
            "angle_sublines", "score_sublines", "mat_klines2sublines")


def plumbing():
    """Fixtures of tests/golden/make_plumbing_golden.py: the reference `Matching` run on the four bundled pairs
    (one file per pair, the point branch in plumbing_points.npz), as one dict."""
    if "plumb" not in _cache:
        names = sorted(f for f in os.listdir(GOLDEN_DIR) if f.startswith("plumbing_pairs_p") and f.endswith(".npz"))
        _cache["plumb"] = {k: v for f in names + ["plumbing_points.npz"]
                           for k, v in np.load(os.path.join(GOLDEN_DIR, f)).items()}
        with open(os.path.join(GOLDEN_DIR, "plumbing_pairs.json")) as f:
            _cache["plumb_meta"] = json.load(f)
    return _cache["plumb"], _cache["plumb_meta"]


def _rebuild_desc(mask_sublines, real, pad):
    """desc_sublines [1,S,T,256] from the real-token descriptors and the shared pad descriptor."""
    mask = mask_sublines[0, :, 1:, 0] > 0
    S, T = mask.shape
    desc = np.broadcast_to(pad.astype(np.float32), (S, T, 256)).copy()
    desc[mask] = real
    return desc[None]


def plumbing_image(npz, prefix):
    """Tokeniser dict (numpy, batch dim 1) of one captured image + the reference's line_desc."""
    d = {k: npz[f"{prefix}_{k}"] for k in TOK_KEYS}
    d["desc_sublines"] = _rebuild_desc(d["mask_sublines"], npz[f"{prefix}_desc_real"], npz[f"{prefix}_desc_pad"])
    return d, npz[f"{prefix}_line_desc"]


def tokenizer_fixture(ci):
    """The reference tokeniser's dict for tokenizer config `ci`, except `desc_sublines` (see check_tokenizer_desc)."""
    if "tok" not in _cache:
        _cache["tok"] = dict(np.load(os.path.join(GOLDEN_DIR, "tokenizer_outputs.npz")))
    npz = _cache["tok"]
    return {k[len(f"c{ci}_"):]: v for k, v in npz.items() if k.startswith(f"c{ci}_") and not k.startswith(f"c{ci}_desc_")}


def check_tokenizer_desc(got, ci, tol=None):
    """`desc_sublines` of tokenizer config `ci` against the reference's: float32 of the same shape, and bit-identical
    (the SHA-256 of all its bytes) or, with `tol`, the stored sample of token rows within tol."""
    import hashlib
    tokenizer_fixture(ci)
    npz = _cache["tok"]
    got = np.ascontiguousarray(got)
    assert got.dtype == np.float32 and got.shape == tuple(npz[f"c{ci}_desc_shape"])
    if tol is None:
        assert hashlib.sha256(got.tobytes()).digest() == npz[f"c{ci}_desc_sha256"].tobytes()
    else:
        rows = got.reshape(-1, got.shape[-1])[npz[f"c{ci}_desc_rows"]]
        assert np.abs(rows - npz[f"c{ci}_desc_sample"]).max() < tol


def matching_line_branch(get_dist_matrix, subline2keyline, nn_matcher_distmat, line_desc0, line_desc1, A0, A1, thr):
    """The line branch of the reference's Matching.forward (models/matching.py:77-81), parameterised by
    the three functions it calls, so that tests can run it over the plugin or over the oracle."""
    distance_sublines = get_dist_matrix(line_desc0, line_desc1)[0]
    distance_matrix = subline2keyline(distance_sublines, A0, A1)
    match_mat = nn_matcher_distmat(distance_matrix, thr, True)
    return match_mat, distance_matrix


def decisive_rows(dist, thr, margin):
    """Rows of [K0,K1] distances whose decision does not hinge on differences below `margin`."""
    d = np.clip(np.asarray(dist, dtype=np.float64), 0.0, None)
    K0, K1 = d.shape
    srt = np.sort(d, axis=1)
    row_gap = srt[:, 1] - srt[:, 0] if K1 > 1 else np.full(K0, np.inf)
    idx = d.argmin(axis=1)
    csrt = np.sort(d, axis=0)
    col_gap = (csrt[1] - csrt[0]) if K0 > 1 else np.full(K1, np.inf)
    return (row_gap > margin) & (np.abs(srt[:, 0] - thr) > margin) & (col_gap[idx] > margin)
