"""Fixtures that let the checkpoint-dependent tests run from the repository alone.  Needs a checkout of the
reference (yosungho/LineTR) with its shipped checkpoint; imports it read-only and runs it on CPU:

    python tests/golden/make_standin_golden.py <reference checkout>

Writes
  * checkpoint_stats.json: [mean, std, min, max] of every tensor of models/weights/LineTR_weight.pth, from
    which tests/helpers.standin_weights() regenerates a seeded stand-in checkpoint;
  * standin_outputs.npz|json: the reference's LineTransformer forward + line matching with the stand-in on the
    seeded inputs of the shipped-checkpoint cases `real_*` (16 x 21, a 128-line pair, 256 x 32, ragged 512 x 64) and
    on the tokeniser dicts of the four bundled image pairs (plumbing_pairs.npz).  Descriptor sets wider than 16 lines
    are stored as a seeded sample of 8 or 16 lines (`<name>_cols`), distance matrices as a sample of 8 rows, with the
    rows whose match decision no difference below 1e-5 can flip (`p<i>_decisive`);
  * reference_init.json: key order, shapes, float64 sums and sampled values of the reference's random init
    (torch.manual_seed(0), two descriptive layers) and its config.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
torch.set_grad_enabled(False)


def sample_cols(n, k, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return np.sort(rng.choice(n, size=min(k, n), replace=False)).astype(np.int64)


def main(ref):
    sys.path.insert(0, ref)
    from models.line_transformer import LineTransformer as RefLT
    from models.line_process import get_dist_matrix as ref_get_dist_matrix
    from models.nn_matcher import nn_matcher_distmat as ref_nn_matcher_distmat
    from linetr_b200 import synthetic as syn
    from tests import helpers as H

    shipped = torch.load(os.path.join(ref, "models", "weights", "LineTR_weight.pth"), map_location="cpu")
    stats = {k: [float(v.double().mean()), float(v.double().std()) if v.numel() > 1 else 0.0,
                 float(v.double().min()), float(v.double().max())] for k, v in shipped.items()}
    with open(os.path.join(HERE, "checkpoint_stats.json"), "w") as f:
        json.dump(stats, f, indent=0)
    H._cache.clear()
    sd = H.standin_weights()
    model = RefLT({"mode": "train"})
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd.items()})
    model.eval()

    def forward(d):
        return model({k: torch.from_numpy(v.copy()) for k, v in d.items()})["line_desc"].numpy()

    def match(d0, d1, a, b, thr):
        return H.matching_line_branch(ref_get_dist_matrix, model.subline2keyline,
                                      lambda dk, t, m: ref_nn_matcher_distmat(dk, t, is_mutual_NN=m),
                                      d0, d1, torch.from_numpy(a["mat_klines2sublines"][0]),
                                      torch.from_numpy(b["mat_klines2sublines"][0]), thr)

    out, meta = {}, {"torch": torch.__version__, "numpy": np.__version__, "weights": "standin", "cases": {}}

    def put(name, desc, k, seed):
        cols = sample_cols(desc.shape[-1], k, seed)
        out[name], out[f"{name}_cols"] = np.ascontiguousarray(desc[..., cols]), cols

    for name, c in {"real_enc_L16_T21": dict(seed=61, L=16, T=21, ntok=(3, 21)),
                    "real_enc_L256_T32": dict(seed=71, L=256, T=32, ntok=None),
                    "real_enc_L512_T64_ragged": dict(seed=72, L=512, T=64, ntok=(3, 64))}.items():
        d = H.case_inputs(c)
        put(name, forward(d), 16, c["seed"])
        meta["cases"][name] = {**c, "checksum": H.checksum(d)}

    c = dict(seed=62, L=128, T=21, thr=0.8)
    a, b, _ = syn.make_pair_inputs(c["seed"], c["L"], c["T"])
    d0, d1 = forward(a), forward(b)
    mat, _ = match(d0, d1, a, b, c["thr"])
    put("real_pair_L128_d0", d0, 16, 620)
    put("real_pair_L128_d1", d1, 16, 621)
    out["real_pair_L128_mat_idx"] = np.where(mat[0].sum(1) > 0, mat[0].argmax(1), -1).astype(np.int32)
    meta["cases"]["real_pair_L128"] = {**c, "checksum0": H.checksum(a), "checksum1": H.checksum(b), "n_matches": int(mat.sum())}

    npz, pmeta = H.plumbing()
    for p in range(len(pmeta["pairs"])):
        a, _ = H.plumbing_image(npz, f"p{p}_0")
        b, _ = H.plumbing_image(npz, f"p{p}_1")
        d0, d1 = forward(a), forward(b)
        mat, dk = match(d0, d1, a, b, 0.8)
        put(f"p{p}_0_line_desc", d0, 8, 100 + 2 * p)
        put(f"p{p}_1_line_desc", d1, 8, 101 + 2 * p)
        rows = sample_cols(dk.shape[1], 8, 200 + p)
        out[f"p{p}_scores_l"], out[f"p{p}_scores_l_rows"] = np.ascontiguousarray(dk[0][rows]), rows
        out[f"p{p}_matches_l"] = np.where(mat[0].sum(1) > 0, mat[0].argmax(1), -1).astype(np.int32)
        out[f"p{p}_decisive"] = H.decisive_rows(dk[0], 0.8, 1e-5)
        meta["cases"][f"plumbing_p{p}"] = {"n_matches_l": int(mat.sum()), "decisive": int(out[f"p{p}_decisive"].sum()),
                                           "K0": int(dk.shape[1]), "K1": int(dk.shape[2])}
    np.savez_compressed(os.path.join(HERE, "standin_outputs.npz"), **out)
    with open(os.path.join(HERE, "standin_outputs.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)

    torch.manual_seed(0)
    r = RefLT({"mode": "train", "n_line_descriptive_layers": 2})
    init = {"config": r.config, "tensors": []}
    for i, (k, v) in enumerate(r.state_dict().items()):
        flat = v.detach().reshape(-1).double().numpy()
        idx = sample_cols(flat.size, 4, i)
        init["tensors"].append({"key": k, "shape": list(v.shape), "dtype": str(v.dtype), "sum": float(flat.sum()),
                                "idx": idx.tolist(), "values": flat[idx].tolist()})
    with open(os.path.join(HERE, "reference_init.json"), "w") as f:
        json.dump(init, f, indent=0)
    print({k: v.get("n_matches", v.get("n_matches_l")) for k, v in meta["cases"].items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(os.path.abspath(sys.argv[1]))
