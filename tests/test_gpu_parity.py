"""GPU parity tests: the CUDA path (through the C ABI) against the numpy oracle, the committed
reference outputs (tests/golden) and size-independent properties at full BASELINE sizes.

Tolerances: descriptors 1e-3 abs (BASELINE.json north_star; we assert a 10x tighter 1e-4
where the path is fp32 end to end), match indices bit-exact."""
import numpy as np
import pytest
import torch

from linetr_b200 import _native as N
from linetr_b200 import _ops, engine, synthetic as syn
from linetr_b200 import nn_matcher as nnm
from linetr_b200.line_process import get_dist_matrix
from linetr_b200.line_transformer import LineTransformer
from oracle import linetr_oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu
DESC_TOL = 1e-3          # the contract
DESC_TOL_TIGHT = 2e-4    # what we hold ourselves to
DIST_TOL = 2e-5          # distances come from a 3-term split-bf16 tensor-core product (|error| <~ 1.2e-5 on 2 - 2s);
                         # every argmin / threshold decision closer than 1e-4 is re-taken with fp32 FMAs (match_tc.cuh)
DEV = torch.device("cuda", 0)
_models = {}


def model_for(tag):
    if tag not in _models:
        if tag == "standin":
            sd = H.standin_weights()
            nd = 1
        else:
            sd = H.weights_for(tag)
            nd = int(tag.split(":")[2])
        m = LineTransformer({"mode": "train", "n_line_descriptive_layers": nd})
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
        _models[tag] = (m.eval().to(DEV), sd)
    return _models[tag]


def to_dev(d):
    return {k: torch.from_numpy(v).to(DEV) for k, v in d.items()}


def fwd(model, data_np):
    return model(to_dev(data_np))["line_desc"].cpu().numpy()


# ------------------------------------------------------------------ GEMM engine
@pytest.mark.parametrize("M,N_,K,act", [(1, 64, 16, 0), (127, 256, 128, 1), (300, 768, 256, 0), (513, 1024, 256, 2),
                                        (64, 256, 1024, 0), (2816, 256, 256, 0)])
def test_linear_engine_vs_torch_fp32(M, N_, K, act):
    g = torch.Generator().manual_seed(M * 7 + K)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N_, K, generator=g) / K ** 0.5
    b = torch.randn(N_, generator=g)
    r = torch.randn(M, N_, generator=g)
    want = torch.nn.functional.linear(x.double(), w.double(), b.double())
    want = [want, torch.relu(want), torch.nn.functional.gelu(want)][act] + r.double()
    got = _ops.linear(x.to(DEV), w.to(DEV), b.to(DEV), r.to(DEV), act).cpu().double()
    assert (got - want).abs().max().item() < 2e-5


@pytest.mark.parametrize("M,N_,K,act,bn", [(1, 128, 64, 0, 0), (128, 128, 64, 0, 128), (127, 256, 128, 1, 256),
                                           (300, 768, 256, 0, 256), (513, 1024, 256, 2, 0), (64, 256, 1024, 0, 128),
                                           (40000, 256, 256, 0, 256), (20000, 512, 512, 1, 0), (1000, 256, 512, 0, 128),
                                           (700, 64, 128, 1, 64), (3000, 192, 256, 0, 0), (20000, 256, 256, 2, 64)])
def test_persistent_image_gemm_vs_fp64(M, N_, K, act, bn):
    """gemm_img engine: TMA-fed split-bf16 tile images in, fp32 rows + split-bf16 image out,
    persistent CTAs with double-buffered TMEM accumulators (more tiles than SMs at M=40000)."""
    g = torch.Generator().manual_seed(M * 7 + K + N_)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N_, K, generator=g) / K ** 0.5
    b = torch.randn(N_, generator=g)
    r = torch.randn(M, N_, generator=g)
    want = torch.nn.functional.linear(x.double(), w.double(), b.double())
    want = [want, torch.relu(want), torch.nn.functional.gelu(want)][act] + r.double()
    y, y_img = _ops.linear_img(x.to(DEV), w, b.to(DEV), r.to(DEV), act, bn)
    assert (y.cpu().double() - want).abs().max().item() < 1e-4
    assert (y_img.cpu().double() - want).abs().max().item() < 2e-4     # + split-bf16 re-quantisation of the output


# ------------------------------------------------------------------ encoder
@pytest.mark.parametrize("M,K,norm,with_res,with_add", [(300, 256, 1, False, False), (1000, 1024, 1, True, True),
                                                         (128 * 150 + 17, 256, 1, True, False), (777, 256, 2, False, False),
                                                         (128 * 149, 256, 2, False, False)])
def test_row_norm_epilogue_vs_fp64(M, K, norm, with_res, with_add):
    """GEMM with the LayerNorm / L2-normalising epilogue (fc+LN1, w_2+LN2+line pos, final_proj+normalize)."""
    g = torch.Generator().manual_seed(M + K + norm)
    x = torch.randn(M, K, generator=g) * 0.7 + 0.1
    w = torch.randn(256, K, generator=g) / K ** 0.5
    b = torch.randn(256, generator=g) * 0.3
    res = torch.randn(M, 256, generator=g) if with_res else None
    add = torch.randn(M, 256, generator=g) if with_add else None
    gamma, beta = torch.rand(256, generator=g) + 0.5, torch.randn(256, generator=g) * 0.2
    cu = lambda t: t.to(DEV) if t is not None else None
    y, y2 = _ops.linear_img_norm(cu(x), w, cu(b), cu(res), norm, 1e-6, cu(gamma), cu(beta), cu(add))
    pre = x.double() @ w.double().T + b.double()
    if res is not None:
        pre = pre + res.double()
    if norm == 1:
        mu = pre.mean(1, keepdim=True)
        var = ((pre - mu) ** 2).mean(1, keepdim=True)
        want = (pre - mu) / torch.sqrt(var + 1e-6) * gamma.double() + beta.double()
        if add is not None:
            want = want + add.double()
    else:
        want = pre / pre.norm(dim=1, keepdim=True).clamp_min(1e-12)
    assert (y.cpu().double() - want).abs().max() < 2e-5 * max(1.0, float(want.abs().max()))
    assert (y2.cpu().double() - want).abs().max() < 4e-5 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("name", H.ENC_CASES)
def test_forward_vs_reference_golden_and_oracle(name):
    npz, meta = H.golden()
    case = meta["cases"][name]
    model, sd = model_for(case["weights"])
    data = H.case_inputs(case)
    got = fwd(model, data)
    assert got.shape == npz[name].shape
    assert np.abs(got - npz[name]).max() < DESC_TOL_TIGHT           # committed reference output
    assert np.abs(got - orc.line_transformer_forward(sd, data)).max() < DESC_TOL_TIGHT
    assert np.abs(np.linalg.norm(got, axis=1) - 1).max() < 1e-5


@pytest.mark.parametrize("name", H.FULL_CASES)
def test_forward_full_size_vs_reference_golden(name):
    """Full-size images (256 lines x 32 tokens; 512 lines x 64 tokens, ragged token counts) with the shipped
    checkpoint's stand-in against outputs of the unmodified reference committed under tests/golden/ (a sample
    of lines) and against the oracle (all lines)."""
    npz, meta = H.standin()
    case = meta["cases"][name]
    model, sd = model_for("standin")
    data = H.case_inputs(case)
    H.assert_checksum(data, case["checksum"])
    got = fwd(model, data)
    want, got_s = H.sampled(npz, name, got)
    assert got_s.shape == want.shape
    assert np.abs(got_s - want).max() < DESC_TOL_TIGHT
    assert np.abs(got - orc.line_transformer_forward(sd, data)).max() < DESC_TOL_TIGHT
    assert np.abs(np.linalg.norm(got, axis=1) - 1).max() < 1e-5


def test_forward_batched_and_inplace_contract():
    npz, meta = H.golden()
    case = meta["cases"]["enc_B2_L12_T21"]
    model, _ = model_for(case["weights"])
    data = to_dev(H.stack([syn.make_image_inputs(s, case["L"], case["T"], tuple(case["ntok"])) for s in case["seeds"]]))
    before = {k: v.clone() for k, v in data.items()}
    out = model(data)
    assert out is data and "line_desc" in data            # same dict object, updated in place
    for k, v in before.items():
        assert torch.equal(v, data[k]), f"forward mutated input {k}"
    assert tuple(data["line_desc"].shape) == (2, 256, 12) and data["line_desc"].is_cuda
    assert np.abs(data["line_desc"].cpu().numpy() - npz["enc_B2_L12_T21"]).max() < DESC_TOL_TIGHT


def test_mask_is_dead_and_padding_is_live():
    """SURVEY §0 fact 3: the token mask cannot change the output, the content of padded
    token slots does (they are attended to as real keys)."""
    model, sd = model_for("synthetic:0:1")
    d = syn.make_image_inputs(77, 10, 21, (3, 10))
    base = fwd(model, d)
    d2 = {k: v.copy() for k, v in d.items()}
    d2["mask_sublines"] = np.ones_like(d["mask_sublines"])
    assert np.array_equal(fwd(model, d2), base)
    d3 = {k: v.copy() for k, v in d.items()}
    d3["desc_sublines"][0, :, 11:] = -d3["desc_sublines"][0, :, 11:]      # only slots the mask marks as padding
    got = fwd(model, d3)
    assert np.abs(got - base).max() > 1e-4      # far above fp32 noise (~1e-6): padding is attended to
    assert np.abs(got - orc.line_transformer_forward(sd, d3)).max() < DESC_TOL_TIGHT


def test_varlen_batch_equals_per_image():
    """Images with different line counts in one call (cu_lines) == one call per image;
    zero-padding would change the result (SURVEY §0 fact 6)."""
    model, sd = model_for("synthetic:0:1")
    ims = [syn.make_image_inputs(100 + i, L, 21, (2, 21)) for i, L in enumerate((7, 33, 1, 150, 64))]
    eng = engine.PairEngine(model, DEV)
    batch = engine.LineBatch.from_images(ims).to(DEV)
    rows, cf = eng.encode(batch, want_cf=True)
    rows, cf = rows.cpu().numpy(), cf.cpu().numpy()
    for i, im in enumerate(ims):
        want = orc.line_transformer_forward(sd, im)[0]          # [256, L]
        s, e = batch.cu_lines[i], batch.cu_lines[i + 1]
        assert np.abs(rows[s:e].T - want).max() < DESC_TOL_TIGHT
        assert np.abs(cf[256 * s:256 * e].reshape(256, e - s) - want).max() < DESC_TOL_TIGHT


def test_weight_update_repacks():
    model, sd = model_for("synthetic:0:1")
    m = LineTransformer({"mode": "train"})
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.eval().to(DEV)
    d = syn.make_image_inputs(9, 6, 21)
    a = fwd(m, d)
    sd2 = syn.make_state_dict(1, 1)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd2.items()})
    b = fwd(m, d)
    assert np.abs(b - orc.line_transformer_forward(sd2, d)).max() < DESC_TOL_TIGHT
    assert np.abs(a - b).max() > 1e-2


# ------------------------------------------------------------------ matcher
def test_nn_matcher_golden_exact():
    npz, _ = H.golden()
    e0, e1, _ = syn.make_descriptor_pair(51, 64, 48)
    for mutual in (True, False):
        mat, dist = nnm.nn_matcher(e0, e1, 0.8, mutual)
        assert mat.dtype == np.float64 and mat.shape == (1, 64, 48) and dist.dtype == np.float32
        assert np.array_equal(mat, npz[f"nn_64_48_mat_m{int(mutual)}"])
        assert np.abs(dist - npz["nn_64_48_dist"]).max() < DIST_TOL
    mat, _ = nnm.nn_matcher(e0, e1, 0.05, True)
    assert np.array_equal(mat, npz["nn_64_48_mat_thr005"])


def test_distmat_ties_clip_threshold_exact():
    npz, _ = H.golden()
    for mutual in (True, False):
        got = nnm.nn_matcher_distmat(npz["distmat_ties_in"], 0.5, mutual)
        assert np.array_equal(got, npz[f"distmat_ties_mat_m{int(mutual)}"])


@pytest.mark.parametrize("n0,n1", [(1, 1), (1, 40), (33, 1), (257, 300), (1000, 999)])
def test_distmat_random_vs_oracle_exact(n0, n1):
    rng = np.random.Generator(np.random.PCG64(n0 * 1000 + n1))
    # quantised values -> many exact ties; some negatives -> clip
    d = (rng.integers(-2, 40, size=(1, n0, n1)) / 16.0).astype(np.float32)
    for mutual in (True, False):
        for thr in (0.5, 0.0, 10.0):
            assert np.array_equal(nnm.nn_matcher_distmat(d, thr, mutual), orc.nn_matcher_distmat(d, thr, mutual))


def test_get_dist_matrix_and_s2k_golden():
    npz, meta = H.golden()
    c = meta["cases"]["s2k"]
    f0, f1, _ = syn.make_descriptor_pair(c["seed"], sum(c["nsub0"]), sum(c["nsub1"]))
    dist = get_dist_matrix(f0[None], f1[None])
    assert dist.dtype == np.float32 and np.abs(dist[0] - npz["s2k_dist_sub"]).max() < DIST_TOL

    def adj(ns):
        A = np.zeros((len(ns), sum(ns)), dtype=np.float32)
        s = 0
        for i, n in enumerate(ns):
            A[i, s:s + n] = 1.0 / n
            s += n
        return torch.from_numpy(A)
    m = LineTransformer({"mode": "train"})
    dk = m.subline2keyline(npz["s2k_dist_sub"], adj(c["nsub0"]), adj(c["nsub1"]))
    assert dk.shape == npz["s2k_dist_key"].shape and np.abs(dk - npz["s2k_dist_key"]).max() < 2e-6
    assert np.array_equal(nnm.nn_matcher_distmat(dk, 0.8, True), npz["s2k_mat"])
    eye = m.subline2keyline(npz["s2k_dist_sub"], torch.eye(sum(c["nsub0"])), torch.eye(sum(c["nsub1"])))
    assert np.array_equal(eye[0], npz["s2k_dist_sub"])


def test_pair_pipeline_vs_reference_golden():
    npz, meta = H.golden()
    case = meta["cases"]["pair_L32_27"]
    model, sd = model_for(case["weights"])
    a, b, _ = syn.make_pair_inputs(case["seed"], case["L0"], case["T"], n_lines1=case["L1"],
                                   n_real_tokens=tuple(case["ntok"]))
    eng = engine.PairEngine(model, DEV)
    res = eng.match_pairs(engine.LineBatch.from_images([a]).to(DEV), engine.LineBatch.from_images([b]).to(DEV),
                          case["thr"], keep_desc=True, want_dist=True)
    want_idx = orc.match_indices(npz["pair_L32_27_mat"])
    assert np.array_equal(res.pair(0).cpu().numpy(), want_idx)
    assert int(res.counts[0]) == case["n_matches"]
    assert np.abs(res.desc0.cpu().numpy().T - npz["pair_L32_27_d0"][0]).max() < DESC_TOL_TIGHT
    dist = res.dist[:32 * 27].view(32, 27).cpu().numpy()
    assert np.abs(dist - npz["pair_L32_27_dist"][0]).max() < 1e-3


def test_pair_batch_with_keyline_merging_vs_oracle():
    """Several pairs at once, ragged line counts, some key lines split into sublines."""
    model, sd = model_for("synthetic:0:1")
    rng = np.random.Generator(np.random.PCG64(5))
    pairs = []
    for p in range(3):
        L = int(rng.integers(12, 40))
        a, b, _ = syn.make_pair_inputs(200 + p, L, 21, n_lines1=L - int(rng.integers(0, 4)))
        for side in (a, b):
            S = side["desc_sublines"].shape[1]
            ns, left = [], S
            while left > 0:
                n = int(min(left, rng.integers(1, 4)))
                ns.append(n)
                left -= n
            A = np.zeros((len(ns), S), np.float32)
            s = 0
            for i, n in enumerate(ns):
                A[i, s:s + n] = 1.0 / n
                s += n
            side["mat_klines2sublines"] = A[None]
        pairs.append((a, b))
    eng = engine.PairEngine(model, DEV)
    res = eng.match_pairs(engine.LineBatch.from_images([a for a, _ in pairs]).to(DEV),
                          engine.LineBatch.from_images([b for _, b in pairs]).to(DEV), 0.8, want_dist=True)
    for p, (a, b) in enumerate(pairs):
        mat, dk, _, _ = orc.match_pair(sd, a, b, 0.8)
        assert np.array_equal(res.pair(p).cpu().numpy(), orc.match_indices(mat)), f"pair {p}"
        assert int(res.counts[p]) == int(mat.sum())
        K0, K1 = dk.shape[1:]
        got = res.dist[p * res.stride:p * res.stride + K0 * K1].view(K0, K1).cpu().numpy()
        assert np.abs(got - dk[0]).max() < 1e-3


def test_match_packed_equals_match_pairs():
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    for uniform in (True, False):
        pairs = []
        for p in range(3):
            L = 40 if uniform else 20 + 7 * p
            a, b, _ = syn.make_pair_inputs(400 + p, L, 21, n_lines1=L if uniform else L - p)
            pairs.append((a, b))
        r1 = eng.match_pairs(engine.LineBatch.from_images([a for a, _ in pairs]).to(DEV),
                             engine.LineBatch.from_images([b for _, b in pairs]).to(DEV), 0.8)
        r2 = eng.match_packed(engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).to(DEV), 3, 0.8)
        assert torch.equal(r1.matches0, r2.matches0) and torch.equal(r1.counts, r2.counts)
        for p, (a, b) in enumerate(pairs):
            mat, _, _, _ = orc.match_pair(sd, a, b, 0.8)
            assert np.array_equal(r2.pair(p).cpu().numpy(), orc.match_indices(mat))


def test_host_pipelined_entry_equals_resident():
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    pairs = [syn.make_pair_inputs(500 + p, 16 + 5 * p, 21, n_lines1=16 + 4 * p)[:2] for p in range(5)]
    host = engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).pin()
    want = eng.match_packed(host.to(DEV), 5, 0.8)
    for chunks in (1, 2, 5):
        m0, cnt, off = eng.match_packed_host(host, 5, 0.8, n_chunks=chunks)
        torch.cuda.synchronize()
        assert torch.equal(m0, want.matches0) and torch.equal(cnt, want.counts)
        assert np.array_equal(off, want.offsets0)


def test_concurrent_streams_share_one_model():
    """Two groups of pairs encoded + matched on two CUDA streams at the same time through ONE model
    handle give exactly the serial results (the encode workspace is per stream)."""
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    groups = []
    for g in range(2):
        pairs = [syn.make_pair_inputs(700 + 100 * g + p, 128, 21)[:2] for p in range(24)]
        groups.append(engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).to(DEV))
    want = [eng.match_packed(b, 24, 0.8, keep_desc=True) for b in groups]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in groups]
    for _ in range(3):
        got = []
        for b, s in zip(groups, streams):
            with torch.cuda.stream(s):
                got.append(eng.match_packed(b, 24, 0.8, keep_desc=True))
        torch.cuda.synchronize()
        for w, r in zip(want, got):
            assert torch.equal(w.desc0, r.desc0) and torch.equal(w.desc1, r.desc1)
            assert torch.equal(w.matches0, r.matches0) and torch.equal(w.counts, r.counts)


def test_shipped_checkpoint_cfg1_pair():
    """The shipped checkpoint's stand-in (its per-tensor magnitudes): the reference's outputs (a sample of lines)
    and the oracle (all lines)."""
    npz, meta = H.standin()
    model, sd = model_for("standin")
    case = meta["cases"]["real_enc_L16_T21"]
    want, got = H.sampled(npz, "real_enc_L16_T21", fwd(model, H.case_inputs(case)))
    assert np.abs(got - want).max() < DESC_TOL_TIGHT
    case = meta["cases"]["real_pair_L128"]
    a, b, _ = syn.make_pair_inputs(case["seed"], case["L"], case["T"])
    eng = engine.PairEngine(model, DEV)
    res = eng.match_pairs(engine.LineBatch.from_images([a]).to(DEV), engine.LineBatch.from_images([b]).to(DEV),
                          case["thr"], keep_desc=True)
    _, _, o0, o1 = orc.match_pair(sd, a, b, case["thr"])
    for name, d, o in (("real_pair_L128_d0", res.desc0, o0), ("real_pair_L128_d1", res.desc1, o1)):
        d = d.cpu().numpy().T[None]
        want, got = H.sampled(npz, name, d)
        assert np.abs(got - want).max() < DESC_TOL_TIGHT
        assert np.abs(d - o).max() < DESC_TOL_TIGHT
    assert np.array_equal(res.pair(0).cpu().numpy(), npz["real_pair_L128_mat_idx"])
    assert int(res.counts[0]) == case["n_matches"]


# ------------------------------------------------------------------ full-size properties
@pytest.mark.parametrize("L,T,P", [(128, 21, 8), (256, 32, 4)])
def test_full_size_properties(L, T, P):
    """BASELINE cfg[1]/cfg[2] shapes: unit norm, line-permutation equivariance of the encoder,
    and the matcher recovering the known permutation between the two sides."""
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    sides, perms = ([], []), []
    for p in range(P):
        a, b, perm = syn.make_pair_inputs(300 + p, L, T)
        sides[0].append(a)
        sides[1].append(b)
        perms.append(perm)
    b0 = engine.LineBatch.from_images(sides[0]).to(DEV)
    b1 = engine.LineBatch.from_images(sides[1]).to(DEV)
    res = eng.match_pairs(b0, b1, 0.8, keep_desc=True)
    d0 = res.desc0.cpu().numpy()
    assert np.abs(np.linalg.norm(d0, axis=1) - 1).max() < 1e-5
    # one pair against the oracle at full size
    mat, _, o0, _ = orc.match_pair(sd, sides[0][0], sides[1][0], 0.8)
    assert np.abs(d0[:L].T - o0[0]).max() < DESC_TOL_TIGHT
    assert np.array_equal(res.pair(0).cpu().numpy(), orc.match_indices(mat))
    # permutation equivariance: shuffling the lines of an image shuffles its descriptors
    rng = np.random.Generator(np.random.PCG64(1))
    shuf = rng.permutation(L)
    im = {k: (v[:, shuf] if k != "mat_klines2sublines" else v) for k, v in sides[0][1].items()}
    ds = eng.encode(engine.LineBatch.from_images([im]).to(DEV)).cpu().numpy()
    assert np.abs(ds - d0[L:2 * L][shuf]).max() < 1e-4
    # side 1 line j is side 0 line perm[j]: a match (i -> j) must satisfy perm[j] == i
    for p in range(P):
        m = res.pair(p).cpu().numpy()
        ok = m >= 0
        assert ok.sum() >= 0.9 * L
        assert np.array_equal(perms[p][m[ok]], np.nonzero(ok)[0])


def test_cfg3_ragged_stress_vs_oracle():
    """BASELINE cfg[3] shape class: ragged 32..512 lines per image, 64 tokens per line (ragged mask),
    several pairs per call.  Descriptors of the smallest/largest images vs the oracle, matches of
    every pair recover the known permutation."""
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    rng = np.random.Generator(np.random.PCG64(33))
    Ls = [32, 512, int(rng.integers(33, 512)), int(rng.integers(33, 512))]
    pairs, perms = [], []
    for p, L in enumerate(Ls):
        a, b, perm = syn.make_pair_inputs(600 + p, L, 64, n_real_tokens=(5, 64))
        pairs.append((a, b))
        perms.append(perm)
    batch = engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).to(DEV)
    res = eng.match_packed(batch, len(Ls), 0.8, keep_desc=True)
    d0 = res.desc0.cpu().numpy()
    for p in (0, 1):   # L = 32 and L = 512 (4 key tiles in the attention kernel)
        s, e = batch.cu_lines[p], batch.cu_lines[p + 1]
        want = orc.line_transformer_forward(sd, pairs[p][0])[0]
        assert np.abs(d0[s:e].T - want).max() < DESC_TOL_TIGHT
    for p, L in enumerate(Ls):
        m = res.pair(p).cpu().numpy()
        ok = m >= 0
        assert ok.sum() >= 0.9 * L and np.array_equal(perms[p][m[ok]], np.nonzero(ok)[0])
        assert int(res.counts[p]) == int(ok.sum())


def test_cfg4_matcher_only_1024_exact():
    """BASELINE cfg[4]: matcher only, 1024 x 1024 x d256.  Indices identical to the oracle
    (numpy fp32 BLAS distance + argmin) and to the known permutation."""
    d0, d1, perm = syn.make_descriptor_pair(71, 1024, 1024)
    mat, dist = nnm.nn_matcher(d0, d1, 0.8, True)
    want, wdist = orc.nn_matcher(d0, d1, 0.8, True)
    assert np.array_equal(mat, want)
    assert np.abs(dist - wdist).max() < DIST_TOL
    idx = orc.match_indices(mat)
    ok = idx >= 0
    assert ok.sum() >= 1000 and np.array_equal(perm[idx[ok]], np.nonzero(ok)[0])


def _f64_match(d0, d1, thr, mutual=True):
    """Matcher decisions from float64 distances of the fp32 descriptors [256, n]: exact ties stay exact
    ties (first index wins), everything else is decided far above any fp32 rounding."""
    dist = np.clip(2.0 - 2.0 * (d0.astype(np.float64).T @ d1.astype(np.float64)), 0.0, None)
    return orc.match_indices(orc.nn_matcher_distmat(dist[None], thr, mutual))


@pytest.mark.parametrize("n0,n1", [(1, 1), (5, 300), (130, 127), (256, 384), (700, 513)])
@pytest.mark.parametrize("layout", ["cf", "rows"])
def test_tc_matcher_exact_ties_and_ragged_tiles(n0, n1, layout):
    """Tensor-core matcher (match_tc_kernel + tail): duplicated descriptors on both sides give EXACT
    ties in rows and columns (np.argmin semantics: lowest index), sizes that are not multiples of the
    128-line tile exercise the padding masks; both descriptor layouts of the C ABI."""
    d0, d1, _ = syn.make_descriptor_pair(9000 + n0 + n1, n0, n1)
    rng = np.random.Generator(np.random.PCG64(n0 * 7 + n1))
    for _ in range(max(1, min(n0, n1) // 6)):          # duplicates -> exact ties
        a, b = rng.integers(0, n1, 2)
        d1[:, a] = d1[:, b]
        a, b = rng.integers(0, n0, 2)
        d0[:, a] = d0[:, b]
    for thr in (0.8, 0.3):
        for mutual in (True, False):
            want = _f64_match(d0, d1, thr, mutual)
            if layout == "cf":
                mat, dist = nnm.nn_matcher(d0, d1, thr, mutual)
                got = orc.match_indices(mat)
                ref = np.clip(2.0 - 2.0 * (d0.astype(np.float64).T @ d1.astype(np.float64)), 0.0, None)
                assert np.abs(dist[0] - ref).max() < DIST_TOL
            else:
                a = torch.from_numpy(np.ascontiguousarray(d0.T)).to(DEV)
                b = torch.from_numpy(np.ascontiguousarray(d1.T)).to(DEV)
                out = _ops.match_descriptors(a, b, N.LAYOUT_ROWS, 1, thr, mutual, n0=n0, n1=n1, want_dist=False)
                got = out["matches0"].cpu().numpy()
                assert out["dist_key"] is None and int(out["counts"][0]) == int((want >= 0).sum())
            assert np.array_equal(got, want), (thr, mutual)


def test_tc_matcher_near_ties_take_the_exact_path():
    """Second-best within 1e-6 of the best (far below the tensor-core product's own error): the tail
    kernel must re-take those decisions with ascending-k fp32 FMAs - indices equal a sequential fp32
    FMA evaluation of the same dot products."""
    n0, n1 = 96, 200
    d0, d1, _ = syn.make_descriptor_pair(4242, n0, n1)
    rng = np.random.Generator(np.random.PCG64(1))
    for j in range(0, n1 - 1, 2):                      # column j+1 = column j nudged by ~1 ulp in a few channels
        d1[:, j + 1] = d1[:, j]
        k = rng.integers(0, 256, 3)
        d1[k, j + 1] = np.nextafter(d1[k, j + 1], np.float32(1.0))
    # sequential fp32 FMA reference (ascending k), the arithmetic the tail kernel promises
    acc = np.zeros((n0, n1), np.float32)
    for k in range(256):
        acc = (acc.astype(np.float64) + d0[k][:, None].astype(np.float64) * d1[k][None, :].astype(np.float64)).astype(np.float32)
    dist = np.maximum(np.float32(2.0) - np.float32(2.0) * acc, np.float32(0.0))
    want = orc.match_indices(orc.nn_matcher_distmat(dist[None], 0.8, True))
    got = orc.match_indices(nnm.nn_matcher(d0, d1, 0.8, True)[0])
    assert np.array_equal(got, want)


def test_tc_matcher_batched_varlen_equals_single_pairs():
    """ltr_match on a ragged batch (cu offsets, pair-aligned tiles) == the same pairs one by one."""
    rng = np.random.Generator(np.random.PCG64(77))
    sizes = [(int(rng.integers(1, 400)), int(rng.integers(1, 400))) for _ in range(5)]
    pairs = [syn.make_descriptor_pair(600 + i, a, b)[:2] for i, (a, b) in enumerate(sizes)]
    d0 = torch.from_numpy(np.concatenate([p[0].T for p in pairs], 0).copy()).to(DEV)
    d1 = torch.from_numpy(np.concatenate([p[1].T for p in pairs], 0).copy()).to(DEV)
    cu0 = np.concatenate([[0], np.cumsum([a for a, _ in sizes])]).astype(np.int32)
    cu1 = np.concatenate([[0], np.cumsum([b for _, b in sizes])]).astype(np.int32)
    out = _ops.match_descriptors(d0, d1, N.LAYOUT_ROWS, len(sizes), 0.8, True, cu0=torch.from_numpy(cu0).to(DEV),
                                 cu1=torch.from_numpy(cu1).to(DEV), max_n0=max(a for a, _ in sizes),
                                 max_n1=max(b for _, b in sizes), want_dist=False)
    m = out["matches0"].cpu().numpy()
    for i, (a, b) in enumerate(pairs):
        want = _f64_match(a, b, 0.8, True)
        assert np.array_equal(m[cu0[i]:cu0[i + 1]], want), i
        assert int(out["counts"][i]) == int((want >= 0).sum())


def test_encoder_tiles_equal_converted_tiles():
    """Uniform 128-line images: the encoder's final GEMM writes the matcher's operand tiles itself
    (match_packed); the result must equal the path that converts the fp32 rows (no tiles given)."""
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    pairs = [syn.make_pair_inputs(880 + p, 128, 21)[:2] for p in range(3)]
    batch = engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs]).to(DEV)
    r = eng.match_packed(batch, 3, 0.8, keep_desc=True)
    out = _ops.match_descriptors(r.desc0, r.desc1, N.LAYOUT_ROWS, 3, 0.8, True, n0=128, n1=128, want_dist=True)
    assert torch.equal(out["matches0"], r.matches0) and torch.equal(out["counts"], r.counts)
    assert r.dist is None and torch.equal(out["scores0"], r.scores0)
    for p, (a, b) in enumerate(pairs):
        mat, _, _, _ = orc.match_pair(sd, a, b, 0.8)
        assert np.array_equal(r.pair(p).cpu().numpy(), orc.match_indices(mat))


@pytest.mark.parametrize("cfg", [{}, {"max_tokens": 8, "token_distance": 12}, {"min_length": 40, "max_keylines": 20}])
def test_gpu_tokenizer_equals_cpu_glue(cfg):
    """ltr_tokenize (GPU) vs the committed outputs of the REFERENCE tokeniser (tests/golden/tokenizer_outputs.npz,
    generated by make_plumbing_golden.py from models/line_process.py:100-196) and vs the CPU glue:
    geometry/masks/adjacency identical, descriptors to fp32 rounding (the reference's: a stored sample of tokens)."""
    from tests.test_tokenizer import CFGS, fake_lines, fake_superpoint
    sp = fake_superpoint(7)
    sp_dev = {k: v.to(DEV) for k, v in sp.items()}
    m = LineTransformer({"mode": "train", **cfg})
    want = m.preprocess(fake_lines(7, 60), (1, 1, 480, 640), sp, None)
    got = m.preprocess(fake_lines(7, 60), (1, 1, 480, 640), sp_dev, None)
    ci = CFGS.index(cfg)
    ref = H.tokenizer_fixture(ci)
    assert set(want.keys()) == set(got.keys()) == set(ref.keys()) | {"desc_sublines"}
    for k in want:
        g = got[k].cpu()
        if k == "desc_sublines":
            assert g.shape == want[k].shape, k
            assert (g - want[k]).abs().max().item() < 2e-6, k
            H.check_tokenizer_desc(want[k].numpy(), ci)
            H.check_tokenizer_desc(g.numpy(), ci, 2e-6)
        else:
            assert g.shape == want[k].shape == ref[k].shape, k
            assert torch.equal(g, want[k]), k
            assert np.array_equal(g.numpy(), ref[k]), k
    # and the tokenised dict drives the encoder
    out = m.eval().to(DEV)(got)["line_desc"]
    assert out.shape[1] == 256 and torch.isfinite(out).all()


@pytest.mark.parametrize("L,T", [(9, 1), (5, 100), (3, 128), (40, 7)])
def test_token_count_extremes_vs_oracle(L, T):
    """Tiles of the fused token kernel hold floor(128 / T) whole lines: T = 1 (128 lines per tile),
    T > 64 (one line per tile) and a T that does not divide 128."""
    model, sd = model_for("synthetic:0:1")
    d = syn.make_image_inputs(800 + T, L, T, (1, T))
    got = fwd(model, d)
    assert np.abs(got - orc.line_transformer_forward(sd, d)).max() < DESC_TOL_TIGHT


def test_c_abi_error_paths():
    """Errors cross the C ABI as negative return codes + ltr_last_error(), never as crashes."""
    import ctypes as C
    model, _ = model_for("synthetic:0:1")
    h = model._get_handle(DEV)
    lib = N.load()
    d = to_dev(syn.make_image_inputs(1, 4, 21))
    flat = lambda k, *s: d[k].reshape(4, *s).contiguous()
    ten = [flat("sublines", 2, 2), flat("resp_sublines", 1), flat("angle_sublines", 2), flat("pnt_sublines", 21, 2),
           flat("desc_sublines", 21, 256), flat("score_sublines", 21, 1)]
    out = torch.empty(4 * 256, device=DEV)
    ws = torch.empty(1024, dtype=torch.uint8, device=DEV)

    def call(n_tokens=21, ws_bytes=1024, lpi=4):
        inp = N.LtrEncodeInput(*[t.data_ptr() for t in ten], None, None, 1, 4, n_tokens, lpi, 640.0, 480.0)
        outp = N.LtrEncodeOutput(out.data_ptr(), None, None)
        return lib.ltr_encode(h.ptr, C.byref(inp), C.byref(outp), C.c_void_p(ws.data_ptr()), ws_bytes, None)
    assert call() == -3 and b"workspace" in lib.ltr_last_error()          # LTR_E_WORKSPACE
    assert call(n_tokens=129) == -4                                        # LTR_E_UNSUPPORTED
    assert call(lpi=3) == -1                                               # LTR_E_INVALID
    with pytest.raises(N.LtrError):
        _ops.ModelHandle({"klenc.cls_token": np.zeros(256, np.float32)}, 0)   # missing checkpoint tensors


# ------------------------------------------------------------------ cfg[0]: the reference Matching's data through the plugin
def _shipped_model(tmp_path_factory):
    if "shipped_test_mode" not in _models:
        # exactly what models/matching.py:16 constructs from match_line_pairs.py's config (mode 'test' loads the
        # checkpoint; here the shipped checkpoint's stand-in)
        p = H.save_standin_checkpoint(tmp_path_factory.mktemp("weights") / "LineTR_weight.pth")
        m = LineTransformer({"max_keylines": -1, "min_length": 16, "token_distance": 8, "nn_threshold": 0.8,
                             "weights_path": p})
        _models["shipped_test_mode"] = m.eval().to(DEV)
    return _models["shipped_test_mode"]


@pytest.mark.parametrize("pair", [0, 1, 2, 3])
def test_plumbing_real_pairs_through_plugin(pair, tmp_path_factory):
    """The tokeniser dicts the UNMODIFIED reference `Matching` built for the four bundled image pairs
    (assets/input_pairs.txt, match_line_pairs.py defaults) replayed through the plugin with the call
    sequence of models/matching.py:41,59,77-81.  Descriptors with the shipped checkpoint's stand-in against
    the reference's with it and the oracle; the line branch on the descriptors the reference computed with the
    shipped checkpoint against what the reference produced from them."""
    npz, meta = H.plumbing()
    snpz, _ = H.standin()
    model = _shipped_model(tmp_path_factory)
    sd = H.standin_weights()
    a, want0 = H.plumbing_image(npz, f"p{pair}_0")
    b, want1 = H.plumbing_image(npz, f"p{pair}_1")
    da, db = to_dev(a), to_dev(b)
    got0 = model(da)["line_desc"].cpu().numpy()
    got1 = model(db)["line_desc"].cpu().numpy()
    for side, got, im in ((0, got0, a), (1, got1, b)):
        want, got_s = H.sampled(snpz, f"p{pair}_{side}_line_desc", got)
        assert np.abs(got_s - want).max() < DESC_TOL_TIGHT
        assert np.abs(got - orc.line_transformer_forward(sd, im)).max() < DESC_TOL_TIGHT
    thr = model.config["nn_threshold"]
    A0, A1 = da["mat_klines2sublines"][0], db["mat_klines2sublines"][0]
    mat, dist = H.matching_line_branch(get_dist_matrix, model.subline2keyline, nnm.nn_matcher_distmat, want0, want1,
                                       A0, A1, thr)
    assert mat.dtype == np.float64 and mat.shape == (1, a["klines"].shape[1], b["klines"].shape[1])
    assert np.abs(dist[0] - npz[f"p{pair}_scores_l"]).max() < DESC_TOL
    got = orc.match_indices(mat)
    want = npz[f"p{pair}_matches_l"]
    # distances agree to <= 1e-3: decisions the reference itself took by a smaller margin than that are not
    # pinned by the 1e-3 contract (none differs in practice - reported below)
    dec = H.decisive_rows(npz[f"p{pair}_scores_l"], thr, 2e-3)
    assert np.array_equal(got[dec], want[dec])
    assert dec.sum() >= 0.9 * len(want)
    assert (got != want).sum() <= 1, f"{(got != want).sum()} of {len(want)} line matches differ from the reference"
    # the batched front-end (key-line merging inside ltr_match) takes the same decisions as the drop-in call sequence
    # wherever the two distance computations (each within DIST_TOL) cannot disagree: the untrained stand-in puts
    # real lines much closer together than the shipped checkpoint does
    mat, dist = H.matching_line_branch(get_dist_matrix, model.subline2keyline, nnm.nn_matcher_distmat, got0, got1,
                                       A0, A1, thr)
    got = orc.match_indices(mat)
    dec = H.decisive_rows(dist[0], thr, 2 * DIST_TOL)
    assert dec.sum() >= 0.6 * len(got)
    eng = engine.PairEngine(model, DEV)
    res = eng.match_pairs(engine.LineBatch.from_images([a]).to(DEV), engine.LineBatch.from_images([b]).to(DEV), thr)
    front = res.pair(0).cpu().numpy()
    assert np.array_equal(front[dec], got[dec])
    assert int(res.counts[0]) == int((front >= 0).sum())


def test_plumbing_point_branch_real_superpoint_descriptors():
    """models/matching.py:69-71: nn_matcher on the SuperPoint descriptors of a real pair (threshold 0.7)."""
    npz, meta = H.plumbing()
    mat, dist = nnm.nn_matcher(npz["p0_desc_pnt0"], npz["p0_desc_pnt1"], 0.7, True)
    assert np.array_equal(orc.match_indices(mat), npz["p0_matches_p"])
    assert int(mat.sum()) == meta["pairs"][0]["n_matches_p"]


# ------------------------------------------------------------------ training-side matcher (evaluations/matcher.py)
def test_eval_matcher_vs_reference_outputs():
    """SURVEY 8f row 4: nn_matcher_batches (dustbin row/column), nn_matcher and nn_matcher_score of the
    reference's evaluations/matcher.py, batched through ltr_match (dist_mode 1: ||a||^2 + ||b||^2 - 2ab on
    tcgen05) - against the committed outputs of the reference functions themselves."""
    import os
    from linetr_b200 import eval_matcher as em
    npz = dict(np.load(os.path.join(H.GOLDEN_DIR, "eval_matcher_outputs.npz")))
    d0, d1 = npz["eval_desc0"], npz["eval_desc1"]
    for mutual in (False, True):
        got = em.nn_matcher_batches(d0, d1, 0.9, mutual)
        assert got.dtype == np.float64 and np.array_equal(got, npz[f"eval_batches_m{int(mutual)}"])
        one = em.nn_matcher(d0[0], d1[0], 0.9, mutual)
        assert one.dtype == np.float32 and np.array_equal(one, npz[f"eval_single_m{int(mutual)}"])
        assert np.array_equal(em.nn_matcher_score(npz["eval_score_in"], 0.5, mutual), npz[f"eval_score_m{int(mutual)}"])
    assert em.nn_matcher_batches(d0[:, :, :0], d1, 0.9, True).shape == (3, 1, 132)


def test_host_pipelined_entry_with_keyline_merging():
    """match_packed_host on a batch whose key lines are split into sublines == match_packed on the device copy."""
    model, sd = model_for("synthetic:0:1")
    eng = engine.PairEngine(model, DEV)
    rng = np.random.Generator(np.random.PCG64(8))
    pairs = []
    for p in range(5):
        L = int(rng.integers(10, 50))
        a, b, _ = syn.make_pair_inputs(1200 + p, L, 21, n_lines1=L - int(rng.integers(0, 3)))
        for side in (a, b):
            S = side["desc_sublines"].shape[1]
            ns, left = [], S
            while left > 0:
                n = int(min(left, rng.integers(1, 4)))
                ns.append(n)
                left -= n
            A = np.zeros((len(ns), S), np.float32)
            s0 = 0
            for i, n in enumerate(ns):
                A[i, s0:s0 + n] = 1.0 / n
                s0 += n
            side["mat_klines2sublines"] = A[None]
        pairs.append((a, b))
    host = engine.LineBatch.from_images([a for a, _ in pairs] + [b for _, b in pairs])
    assert host.sub_off is not None
    want = eng.match_packed(host.to(DEV), 5, 0.8)
    for chunks in (1, 2, 5):
        m0, cnt, off0 = eng.match_packed_host(host.pin(), 5, 0.8, n_chunks=chunks)
        assert torch.equal(m0, want.matches0) and torch.equal(cnt, want.counts)
        assert np.array_equal(off0, want.offsets0)
    for p, (a, b) in enumerate(pairs):
        mat, _, _, _ = orc.match_pair(sd, a, b, 0.8)
        assert np.array_equal(want.pair(p).cpu().numpy(), orc.match_indices(mat))


def test_peer_counts_fused_gather_world2():
    """Multi-GPU (needs >= 2 GPUs on the box): the match counts published to every rank by the matcher's tail
    kernel (multimem.st / peer stores over NVLink, no collective kernel) equal an ncclAllGather of them."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29577", os.path.join(root, "tools", "peer_counts_check.py")],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])


@pytest.mark.parametrize("d_inner,L", [(512, 37), (2048, 20), (384, 9)])
def test_ffn_width_other_than_1024(d_inner, L):
    """config['d_inner'] != 1024 (the reference accepts any): the FFN hidden image of the workspace is sized by
    d_inner and the GEMM launcher checks its k-block ranges (a fixed 1024-wide image used to alias tiles
    silently).  384 is not a multiple of 256: the line stage falls back from the chained engine."""
    sd = syn.make_state_dict(3, 1, d_inner=d_inner)
    m = LineTransformer({"mode": "train", "d_inner": d_inner})
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.eval().to(DEV)
    d = syn.make_image_inputs(900 + d_inner, L, 21, (3, 21))
    want = orc.line_transformer_forward(sd, d)
    assert np.abs(fwd(m, d) - want).max() < DESC_TOL_TIGHT
