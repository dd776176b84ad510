"""cfg[0] plumbing fixtures: run the UNMODIFIED reference `Matching` (models/matching.py) on the four
bundled image pairs (assets/input_pairs.txt) exactly as match_line_pairs.py configures it, on CPU,
and commit what the hot path received and produced.  Needs a checkout of the reference:

    python tests/golden/make_plumbing_golden.py <reference checkout>

The reference's LSD wrapper needs opencv-contrib's `cv2.line_descriptor` (absent here, SURVEY.md 8c):
a TEST-ONLY shim detector built on the main-module `cv2.createLineSegmentDetector` stands in.  Which
lines are detected is irrelevant to hot-path parity - both implementations receive the same tokenised
dict - but the tokeniser, LineTransformer.forward, get_dist_matrix, subline2keyline and
nn_matcher_distmat calls are the reference's own, with real SuperPoint descriptors, real line
geometry, real key-line -> subline splits (mat_klines2sublines is not the identity).

The line transformer keeps the MAX_KEYLINES strongest key lines of each image (the reference's own
`max_keylines` option; every other setting is match_line_pairs.py's), which keeps each fixture file well
under 1 MB.  Stored per image (fixture `plumbing_pairs_p<i>.npz`, one file per pair): the tokeniser dict (descriptors of padded token
slots are all the descriptor sampled at (0, 0), so only real-token descriptors + that one pad
descriptor are stored and `tests/helpers.plumbing_image` rebuilds the tensor bit-exactly) and the
reference outputs `line_desc`, `matches_l`, `matching_scores_l`; for one pair also the SuperPoint point
descriptors + `matches_p` (the nn_matcher call of matching.py:69-71, `plumbing_points.npz`).
Also writes tokenizer fixtures (`tokenizer_outputs.npz`): outputs of the reference tokeniser
(`LineTransformer.preprocess`, models/line_transformer.py:251-275 -> models/line_process.py:100-196) for the seeded
fake detections / fake SuperPoint maps of tests/test_tokenizer.py, so that the GPU tokenizer is
checked against REFERENCE data.  `desc_sublines` is stored as the SHA-256 of its bytes (bit-identity checks),
its shape and DESC_SAMPLE seeded token rows (tolerance checks).
"""
import hashlib
import json
import os
import sys
import types

import cv2
import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
torch.set_grad_enabled(False)
MAX_KEYLINES = 20
DESC_SAMPLE = 64


class ShimKeyLine:
    """The KeyLine fields the reference reads (models/line_process.py:6-20)."""

    def __init__(self, x0, y0, x1, y1, octave=0):
        self.startPointX, self.startPointY, self.endPointX, self.endPointY = float(x0), float(y0), float(x1), float(y1)
        self.lineLength = float(np.hypot(x1 - x0, y1 - y0))
        self.octave = octave


class ShimLSD:
    """Stand-in for models/line_detector.py:11-28 (same constructor / detect_torch surface)."""
    default_config = {"n_octave": 2, "scale": 2}

    def __init__(self, config):
        self.config = {**self.default_config, **config}
        self.lsd = cv2.createLineSegmentDetector(0)

    def detect_torch(self, image):
        img = (image * 255).cpu().numpy().squeeze().astype("uint8")
        lines = self.lsd.detect(img)[0]
        if lines is None:
            return []
        return [ShimKeyLine(*l[0]) for l in lines]


def reference_matching_config():
    """The config dict match_line_pairs.py:54-73 builds (defaults of its argparse), MAX_KEYLINES key lines."""
    return {
        "auto_min_length": True,
        "superpoint": {"nms_radius": 4, "keypoint_threshold": 0.005, "max_keypoints": 1024, "nn_threshold": 0.7},
        "lsd": {"n_octave": 2},
        "linetransformer": {"max_keylines": MAX_KEYLINES, "min_length": 16, "token_distance": 8, "nn_threshold": 0.8},
    }


def read_image(path, resize=(640, 480)):
    """match_line_pairs.py:11-16."""
    image = cv2.imread(str(path), cv2.IMREAD_GRAYSCALE)
    image = cv2.resize(image.astype("float32"), (resize[0], resize[1]))
    return torch.from_numpy(image / 255.).float()[None, None]


TOK_KEYS = ("klines", "length_klines", "angles", "sublines", "pnt_sublines", "mask_sublines", "resp_sublines",
            "angle_sublines", "score_sublines", "mat_klines2sublines")


def pack_image(out, prefix, pred, side):
    """Store the tokeniser dict of one image compactly (see module docstring)."""
    g = lambda k: pred[k + side].numpy()
    for k in TOK_KEYS:
        out[f"{prefix}_{k}"] = g(k)
    desc = g("desc_sublines")[0]                      # [S, T, 256]
    mask = g("mask_sublines")[0, :, 1:, 0] > 0        # [S, T] real-token slots
    pad_rows = desc[~mask]
    if len(pad_rows):
        assert (pad_rows == pad_rows[0]).all(), "padded slots do not share one descriptor"
        out[f"{prefix}_desc_pad"] = pad_rows[0]
    else:
        out[f"{prefix}_desc_pad"] = np.zeros(256, np.float32)
    out[f"{prefix}_desc_real"] = desc[mask]
    out[f"{prefix}_line_desc"] = g("line_desc")


def main(ref):
    sys.path.insert(0, ref)
    import models.matching as ref_matching
    ref_matching.LSD = ShimLSD                       # the only substitution; everything else is stock
    matching = ref_matching.Matching(reference_matching_config()).eval()
    with open(os.path.join(ref, "assets", "input_pairs.txt")) as f:
        pairs = [l.split()[:2] for l in f.readlines() if l.strip()]
    meta = {"pairs": [], "max_keylines": MAX_KEYLINES}
    for i, (n0, n1) in enumerate(pairs):
        out = {}
        im0 = read_image(os.path.join(ref, "assets", n0))
        im1 = read_image(os.path.join(ref, "assets", n1))
        pred = matching({"image0": im0, "image1": im1})
        pack_image(out, f"p{i}_0", pred, "0")
        pack_image(out, f"p{i}_1", pred, "1")
        out[f"p{i}_matches_l"] = np.where(pred["matches_l"][0].numpy().sum(1) > 0,
                                          pred["matches_l"][0].numpy().argmax(1), -1).astype(np.int32)
        out[f"p{i}_scores_l"] = pred["matching_scores_l"][0].numpy()
        info = {"names": [n0, n1], "K0": int(pred["klines0"].shape[1]), "K1": int(pred["klines1"].shape[1]),
                "S0": int(pred["sublines0"].shape[1]), "S1": int(pred["sublines1"].shape[1]),
                "n_matches_l": int(pred["matches_l"].sum()), "n_matches_p": int(pred["matches_p"].sum()),
                "config_after": {k: matching.linetransformer.config[k] for k in ("min_length", "token_distance", "max_tokens")}}
        d = np.clip(pred["matching_scores_l"][0].numpy().astype(np.float64), 0, None)
        srt = np.sort(d, axis=1)
        info["min_top2_gap_rows"] = float((srt[:, 1] - srt[:, 0]).min())
        if i == 0:   # point branch (matching.py:69-71): descriptors [256, N] + the reference's matches
            np.savez_compressed(os.path.join(HERE, "plumbing_points.npz"), p0_desc_pnt0=pred["descriptors0"][0].numpy(),
                                p0_desc_pnt1=pred["descriptors1"][0].numpy(),
                                p0_matches_p=np.where(pred["matches_p"][0].numpy().sum(1) > 0,
                                                      pred["matches_p"][0].numpy().argmax(1), -1).astype(np.int32))
        meta["pairs"].append(info)
        print(info)
        np.savez_compressed(os.path.join(HERE, f"plumbing_pairs_p{i}.npz"), **out)
    meta["torch"] = torch.__version__
    meta["note"] = "reference Matching (CPU) with a cv2.createLineSegmentDetector shim for the LSD wrapper"

    # ---- tokenizer fixtures (reference preprocess on seeded fake detections) ----
    from models.line_transformer import LineTransformer as RefLT
    from tests.test_tokenizer import fake_lines, fake_superpoint
    tok = {}
    cfgs = [{}, {"max_tokens": 8, "token_distance": 12}, {"min_length": 40, "max_keylines": 20}]
    for ci, cfg in enumerate(cfgs):
        ref = RefLT({"mode": "train", **cfg})
        sp = fake_superpoint(7)
        want = ref.preprocess(fake_lines(7, 60), (1, 1, 480, 640), sp, None)
        for k, v in want.items():
            a = v.numpy()
            if k == "desc_sublines":
                a = np.ascontiguousarray(a)
                tok[f"c{ci}_desc_sha256"] = np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)
                tok[f"c{ci}_desc_shape"] = np.array(a.shape, np.int64)
                flat = a.reshape(-1, a.shape[-1])
                rows = np.sort(np.random.Generator(np.random.PCG64(ci)).choice(len(flat), DESC_SAMPLE, replace=False))
                tok[f"c{ci}_desc_rows"], tok[f"c{ci}_desc_sample"] = rows, flat[rows]
            else:
                tok[f"c{ci}_{k}"] = a
    meta["tokenizer_cfgs"] = cfgs

    # ---- training-side matchers (evaluations/matcher.py), seeded descriptor sets with non-unit norms ----
    from evaluations import matcher as ref_eval
    from linetr_b200 import synthetic as syn
    ev = {}
    rng = np.random.Generator(np.random.PCG64(99))
    d0 = np.stack([syn.make_descriptor_pair(700 + i, 150, 131)[0] for i in range(3)])
    d1 = np.stack([syn.make_descriptor_pair(700 + i, 150, 131)[1] for i in range(3)])
    d0 = (d0 * rng.uniform(0.8, 1.25, size=(3, 1, 150))).astype(np.float32)     # per-line norms != 1
    d1 = (d1 * rng.uniform(0.8, 1.25, size=(3, 1, 131))).astype(np.float32)
    ev["eval_desc0"], ev["eval_desc1"] = d0, d1
    for mutual in (False, True):
        ev[f"eval_batches_m{int(mutual)}"] = ref_eval.nn_matcher_batches(d0, d1, 0.9, mutual)
        ev[f"eval_single_m{int(mutual)}"] = ref_eval.nn_matcher(d0[0], d1[0], 0.9, mutual)
    dm = rng.integers(0, 9, size=(40, 37)).astype(np.float32) * np.float32(0.125) - np.float32(0.125)
    ev["eval_score_in"] = dm
    for mutual in (False, True):
        ev[f"eval_score_m{int(mutual)}"] = ref_eval.nn_matcher_score(dm, 0.5, mutual)
    np.savez_compressed(os.path.join(HERE, "eval_matcher_outputs.npz"), **ev)
    np.savez_compressed(os.path.join(HERE, "tokenizer_outputs.npz"), **tok)
    with open(os.path.join(HERE, "plumbing_pairs.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    for fn in sorted(os.listdir(HERE)):
        if fn.endswith(".npz"):
            print(fn, os.path.getsize(os.path.join(HERE, fn)) / 1e6, "MB")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(os.path.abspath(sys.argv[1]))
