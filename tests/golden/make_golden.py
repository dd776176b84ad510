"""Generate golden fixtures by running the UNMODIFIED reference (a checkout of it, imported
read-only) on seeded inputs:

    python tests/golden/make_golden.py <reference checkout>

Inputs and synthetic weights are regenerable from seeds (linetr_b200/synthetic.py), so the
fixtures store only the reference OUTPUTS plus input checksums that detect generator
drift.  The reference is executed on CPU, eval mode, no grad (SURVEY.md §8c/§8d).  The cases with the
shipped checkpoint live in make_standin_golden.py.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.path.abspath(sys.argv[1]) if len(sys.argv) == 2 else sys.exit(__doc__)
sys.path.insert(0, REF)

from linetr_b200 import synthetic as syn  # noqa: E402
from models.line_transformer import LineTransformer as RefLT  # noqa: E402
from models.line_process import get_dist_matrix as ref_get_dist_matrix  # noqa: E402
from models.nn_matcher import nn_matcher as ref_nn_matcher  # noqa: E402
from models.nn_matcher import nn_matcher_distmat as ref_nn_matcher_distmat  # noqa: E402

torch.set_grad_enabled(False)


def checksum(d):
    return {k: float(np.asarray(v, dtype=np.float64).sum()) for k, v in sorted(d.items())}


def ref_model(sd_np, n_desc_layers=1):
    m = RefLT({"mode": "train", "n_line_descriptive_layers": n_desc_layers})
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd_np.items()})
    return m.eval()


def run_forward(model, data_np):
    data = {k: torch.from_numpy(v.copy()) for k, v in data_np.items()}
    return model(data)["line_desc"].numpy()


def stack(images):
    return {k: np.concatenate([im[k] for im in images], axis=0) for k in images[0]}


def main():
    out = {}
    meta = {"torch": torch.__version__, "numpy": np.__version__, "cases": {}}

    # ---- synthetic weights, encoder cases -------------------------------------------------
    sd0 = syn.make_state_dict(0, 1)
    m0 = ref_model(sd0, 1)
    enc_cases = {
        "enc_L16_T21": dict(seed=11, L=16, T=21, ntok=None),
        "enc_L1_T21": dict(seed=12, L=1, T=21, ntok=None),
        "enc_L37_T5_ragged": dict(seed=13, L=37, T=5, ntok=(2, 5)),
        "enc_L24_T32_ragged": dict(seed=14, L=24, T=32, ntok=(5, 32)),
        "enc_L130_T21": dict(seed=15, L=130, T=21, ntok=(3, 21)),
    }
    for name, c in enc_cases.items():
        d = syn.make_image_inputs(c["seed"], c["L"], c["T"], c["ntok"])
        out[name] = run_forward(m0, d)
        meta["cases"][name] = {**{k: v for k, v in c.items()}, "weights": "synthetic:0:1",
                               "checksum": checksum(d)}
    # batched call: two images of equal L in one forward
    ims = [syn.make_image_inputs(21, 12, 21, (4, 21)), syn.make_image_inputs(22, 12, 21, (4, 21))]
    out["enc_B2_L12_T21"] = run_forward(m0, stack(ims))
    meta["cases"]["enc_B2_L12_T21"] = {"seeds": [21, 22], "L": 12, "T": 21, "ntok": (4, 21),
                                       "weights": "synthetic:0:1", "checksum": checksum(stack(ims))}
    # two descriptive layers: only the last one is live (SURVEY.md §0 fact 4)
    sd2 = syn.make_state_dict(5, 2)
    m2 = ref_model(sd2, 2)
    d = syn.make_image_inputs(31, 9, 21, (3, 21))
    out["enc_L9_T21_nd2"] = run_forward(m2, d)
    meta["cases"]["enc_L9_T21_nd2"] = {"seed": 31, "L": 9, "T": 21, "ntok": (3, 21),
                                       "weights": "synthetic:5:2", "checksum": checksum(d)}

    # ---- pair (encode x2 + dist + subline2keyline + mutual NN) -----------------------------
    def run_pair(model, a, b, thr):
        d0 = run_forward(model, a)
        d1 = run_forward(model, b)
        dist = ref_get_dist_matrix(d0, d1)[0]
        dk = model.subline2keyline(dist, torch.from_numpy(a["mat_klines2sublines"][0]),
                                   torch.from_numpy(b["mat_klines2sublines"][0]))
        mat = ref_nn_matcher_distmat(dk, thr, is_mutual_NN=True)
        return d0, d1, dk, mat

    a, b, perm = syn.make_pair_inputs(41, 32, 21, n_lines1=27, n_real_tokens=(4, 21))
    d0, d1, dk, mat = run_pair(m0, a, b, 0.8)
    out["pair_L32_27_d0"], out["pair_L32_27_d1"] = d0, d1
    out["pair_L32_27_dist"], out["pair_L32_27_mat"] = dk, mat
    meta["cases"]["pair_L32_27"] = {"seed": 41, "L0": 32, "L1": 27, "T": 21, "ntok": (4, 21), "thr": 0.8,
                                    "weights": "synthetic:0:1", "checksum0": checksum(a),
                                    "checksum1": checksum(b), "n_matches": int(mat.sum())}

    # ---- matcher only ---------------------------------------------------------------------
    e0, e1, _ = syn.make_descriptor_pair(51, 64, 48)
    for mutual in (True, False):
        mat, dist = ref_nn_matcher(e0, e1, 0.8, is_mutual_NN=mutual)
        out[f"nn_64_48_mat_m{int(mutual)}"] = mat
        out["nn_64_48_dist"] = dist
    mat, _ = ref_nn_matcher(e0, e1, 0.05, is_mutual_NN=True)
    out["nn_64_48_mat_thr005"] = mat
    # distance matrix with exact ties, negatives (clip) and threshold-equal entries
    rng = np.random.Generator(np.random.PCG64(52))
    dm = rng.integers(0, 6, size=(1, 23, 19)).astype(np.float32) * np.float32(0.25) - np.float32(0.25)
    out["distmat_ties_in"] = dm
    for mutual in (True, False):
        out[f"distmat_ties_mat_m{int(mutual)}"] = ref_nn_matcher_distmat(dm, 0.5, is_mutual_NN=mutual)
    # subline2keyline with real segments (line_process.py:163-167 adjacency)
    nsub0, nsub1 = [1, 3, 2, 1, 4], [2, 2, 1, 5]
    def adj(ns):
        A = np.zeros((len(ns), sum(ns)), dtype=np.float32)
        s = 0
        for i, n in enumerate(ns):
            A[i, s:s + n] = 1.0 / n
            s += n
        return A
    A0, A1 = adj(nsub0), adj(nsub1)
    f0, f1, _ = syn.make_descriptor_pair(53, sum(nsub0), sum(nsub1))
    dist = ref_get_dist_matrix(f0[None], f1[None])[0]
    dk = m0.subline2keyline(dist, torch.from_numpy(A0), torch.from_numpy(A1))
    out["s2k_dist_sub"], out["s2k_dist_key"] = dist, dk
    out["s2k_mat"] = ref_nn_matcher_distmat(dk, 0.8, is_mutual_NN=True)
    meta["cases"]["s2k"] = {"seed": 53, "nsub0": nsub0, "nsub1": nsub1}

    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), **out)
    with open(os.path.join(HERE, "reference_outputs.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print("wrote", len(out), "arrays;",
          {k: v.get("n_matches") for k, v in meta["cases"].items() if "n_matches" in v})


if __name__ == "__main__":
    main()
