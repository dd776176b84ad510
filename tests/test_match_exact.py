"""The matcher's exact path (match_exact_kernel): decisions the tensor-core margin test cannot take are re-taken
with ascending-k fp32 FMAs on the whole GPU.  Inputs here are built so that a large share of rows and columns
is ambiguous (best and second-best distance closer than MATCH_EPS = 1e-4), the way the encoder's seeded
weights leave them: near-collapsed descriptors, exact duplicates and 1-ulp nudges.

The reference is a host evaluation of the same arithmetic: every dot product a sequential chain of correctly
rounded fp32 FMAs from 0 (k ascending), then the distance in fp32.  matches0, nn1 and counts must equal it;
scores0 must equal it bit for bit on every row whose reference margin is below MATCH_EPS / 2 (those rows are
certainly on the exact path) and to the tensor-core tolerance elsewhere."""
import numpy as np
import pytest
import torch

from linetr_b200 import _native as N
from linetr_b200 import _ops, synthetic as syn

DEV = torch.device("cuda", 0)
EPS = 1e-4
DIST_TOL = 2e-5
SIZES = [(1, 700), (127, 129), (129, 127), (503, 503), (700, 503), (129, 1)]


def _fma32(x, y, z):
    """Correctly rounded fp32 fma(x, y, z) on arrays (x, y, z float32).  x*y is exact in float64; the float64 sum
    is corrected where rounding it to float32 would round twice (a float32 midpoint hit with a nonzero error)."""
    z64 = z.astype(np.float64)
    p = x.astype(np.float64) * y.astype(np.float64)
    s = z64 + p
    bb = s - z64
    err = (z64 - (s - bb)) + (p - bb)            # s + err == z + x*y exactly (TwoSum)
    r = s.astype(np.float32)
    r64 = r.astype(np.float64)
    need = (s != r64) & (err != 0)
    if need.any():
        other = np.nextafter(r, np.where(s > r64, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
        mid = (r64 + other.astype(np.float64)) * 0.5
        flip = need & (s == mid) & ((err > 0) == (other > r))
        r = np.where(flip, other, r)
    return r


def _ref_dist(a, b, mode, sqa=None, sqb=None):
    """a [..., n0, 256], b [..., n1, 256] float32 -> fp32 distances [..., n0, n1] of the exact path."""
    acc = np.zeros(a.shape[:-1] + b.shape[-2:-1], np.float32)
    for k in range(a.shape[-1]):
        acc = _fma32(a[..., k][..., :, None], b[..., k][..., None, :], acc)
    two = np.float32(2.0)
    if mode == 0:
        d = two - two * acc
    else:
        d = (sqa[..., :, None] + sqb[..., None, :]) - two * acc
    return np.maximum(d, np.float32(0.0)).astype(np.float32)


def _decide(dist, thr, mutual):
    """nn_matcher_distmat on one pair: first-minimum argmins, strict '<' threshold, mutual check."""
    n0, n1 = dist.shape
    if n1 == 0:
        return np.full(n0, -1), np.full(n0, np.inf, np.float32), None
    idx = dist.argmin(1)
    score = dist[np.arange(n0), idx]
    keep = score < np.float32(thr)
    nn1 = dist.argmin(0) if n0 else np.full(n1, -1)
    if mutual:
        keep &= nn1[idx] == np.arange(n0)
    return np.where(keep, idx, -1), score, nn1


def _margin(dist):
    if dist.shape[1] < 2:
        return np.full(dist.shape[0], np.inf)
    s = np.sort(dist, 1)
    return s[:, 1].astype(np.float64) - s[:, 0]


def _unit(x):
    return (x / np.linalg.norm(x.astype(np.float64), axis=1, keepdims=True)).astype(np.float32)


def _collapsed(rng, c, n, s=0.05):
    """unit(c + s * noise) with exact duplicates and 1-ulp nudges of a few channels."""
    x = _unit(c[None, :] + s * rng.standard_normal((n, c.size)))
    for _ in range(n // 8):
        i, j = rng.integers(0, n, 2)
        x[i] = x[j]
        if rng.random() < 0.5:
            k = rng.integers(0, c.size, 3)
            x[i, k] = np.nextafter(x[i, k], np.float32(1.0))
    return x


def _dyadic(rng, base, n):
    """Distance mode 1: small multiples of 2^-7, so every product, norm and distance is exact in fp32 and
    nearby lines are 2^-14 apart - exact ties and sub-MATCH_EPS gaps everywhere."""
    x = np.tile(base, (n, 1))
    for r in range(n):
        k = rng.integers(0, base.size, int(rng.integers(0, 4)))
        x[r, k] += rng.choice([-1, 1], k.size)
    return (x * 2.0 ** -7).astype(np.float32)


def _batch(mode, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    c = rng.standard_normal(256)
    base = rng.integers(-16, 17, 256)
    pairs = []
    for n0, n1 in SIZES:
        if mode == 0:
            pairs.append((_collapsed(rng, c, n0), _collapsed(rng, c, n1)))
        else:
            pairs.append((_dyadic(rng, base, n0), _dyadic(rng, base, n1)))
    return pairs


_refs = {}


def _reference(mode):
    if mode not in _refs:
        pairs = _batch(mode, 31 + mode)
        dists = []
        for a, b in pairs:
            sq = lambda x: (x.astype(np.float64) ** 2).sum(1).astype(np.float32)   # exact for the dyadic inputs
            dists.append(_ref_dist(a, b, mode, *((sq(a), sq(b)) if mode == 1 else ())))
        _refs[mode] = (pairs, dists)
    return _refs[mode]


def _run(pairs, layout, thr, mutual, mode):
    n0s = [a.shape[0] for a, _ in pairs]
    n1s = [b.shape[0] for _, b in pairs]
    cu0 = np.concatenate([[0], np.cumsum(n0s)]).astype(np.int32)
    cu1 = np.concatenate([[0], np.cumsum(n1s)]).astype(np.int32)
    if layout == "rows":
        d0 = np.concatenate([a for a, _ in pairs], 0)
        d1 = np.concatenate([b for _, b in pairs], 0)
        lay = N.LAYOUT_ROWS
    else:   # pair p: [256, n_p] at 256 * first line
        d0 = np.concatenate([a.T.ravel() for a, _ in pairs])
        d1 = np.concatenate([b.T.ravel() for _, b in pairs])
        lay = N.LAYOUT_CHANNEL_FIRST
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    out = _ops.match_descriptors(t(d0), t(d1), lay, len(pairs), thr, mutual, cu0=t(cu0), cu1=t(cu1),
                                 max_n0=max(n0s), max_n1=max(n1s), want_dist=False, dist_mode=mode)
    torch.cuda.synchronize()
    res = {k: out[k].cpu().numpy() for k in ("matches0", "scores0", "nn1", "counts")}
    return res, cu0, cu1


def _check(pairs, dists, res, cu0, cu1, thr, mutual, exact_scores=True):
    for p, dist in enumerate(dists):
        want_m, want_s, want_nn = _decide(dist, thr, mutual)
        m = res["matches0"][cu0[p]:cu0[p + 1]]
        s = res["scores0"][cu0[p]:cu0[p + 1]]
        assert np.array_equal(m, want_m), (p, np.nonzero(m != want_m)[0][:10])
        assert int(res["counts"][p]) == int((want_m >= 0).sum()), p
        if mutual and want_nn is not None and dist.shape[0]:
            assert np.array_equal(res["nn1"][cu1[p]:cu1[p + 1]], want_nn), p
        if dist.shape[1]:
            hard = _margin(dist) < EPS / 2
            if exact_scores:
                assert np.array_equal(s[hard].view(np.uint32), want_s[hard].view(np.uint32)), p
            assert np.abs(s.astype(np.float64) - want_s).max() < DIST_TOL, p


def test_reference_fma_is_correctly_rounded():
    """The host fma emulation against exact rational arithmetic, on random operands and on operands whose float64
    sum rounds onto a float32 midpoint (z in [1, 2), x * y = ulp(z) / 2 * (1 - a^2 2^-46), a < 300)."""
    from fractions import Fraction
    rng = np.random.Generator(np.random.PCG64(5))
    n = 4000
    x = rng.standard_normal(n).astype(np.float32)
    y = rng.standard_normal(n).astype(np.float32)
    z = rng.standard_normal(n).astype(np.float32)
    a = rng.integers(1, 300, n // 2).astype(np.float64)
    x[:n // 2] = (1.0 + a * 2.0 ** -23).astype(np.float32)
    y[:n // 2] = ((1.0 - a * 2.0 ** -23) * 2.0 ** -24).astype(np.float32)
    z[:n // 2] = (1.0 + rng.integers(0, 2 ** 23, n // 2) * 2.0 ** -23).astype(np.float32)
    got = _fma32(x, y, z)
    naive = (z.astype(np.float64) + x.astype(np.float64) * y.astype(np.float64)).astype(np.float32)
    assert (naive != got).sum() > n // 8   # the midpoint cases do round twice without the correction
    for i in range(n):
        exact = Fraction(float(x[i])) * Fraction(float(y[i])) + Fraction(float(z[i]))
        r = np.float32(float(exact))
        lo, hi = (r, np.nextafter(r, np.float32(np.inf))) if Fraction(float(r)) <= exact else (np.nextafter(r, np.float32(-np.inf)), r)
        dl, dh = exact - Fraction(float(lo)), Fraction(float(hi)) - exact
        want = lo if dl < dh or (dl == dh and (lo.view(np.uint32) & 1) == 0) else hi
        assert got[i] == want, i


@pytest.mark.gpu
@pytest.mark.parametrize("mutual", [True, False])
@pytest.mark.parametrize("layout", ["rows", "cf"])
@pytest.mark.parametrize("mode", [0, 1])
def test_collapsed_batch_equals_sequential_fp32(mode, layout, mutual):
    """Ragged batch (1 .. 700 lines) of near-collapsed descriptors: more than 30 % of rows and columns are
    ambiguous; every decision equals the host's sequential fp32 evaluation."""
    pairs, dists = _reference(mode)
    amb_rows = sum(int((_margin(d) < EPS).sum()) for d in dists)
    amb_cols = sum(int((_margin(d.T) < EPS).sum()) for d in dists)
    assert amb_rows > 0.3 * sum(d.shape[0] for d in dists) and amb_cols > 0.3 * sum(d.shape[1] for d in dists)
    thrs = (0.8, 0.005) if mode == 0 else (0.8, 2 * 2.0 ** -14)   # mode 1: a threshold equal to many best distances
    for thr in thrs:
        res, cu0, cu1 = _run(pairs, layout, thr, mutual, mode)
        _check(pairs, dists, res, cu0, cu1, thr, mutual)


@pytest.mark.gpu
def test_one_collapsed_pair_among_separated_pairs():
    """A 512-line collapsed pair in the middle of 63 well-separated 128-line pairs: its ~1000 ambiguous lines are
    the whole work list.  Decisions of every pair are right, and the exact kernel is one launch."""
    rng = np.random.Generator(np.random.PCG64(8))
    c = rng.standard_normal(256)
    pairs = []
    for p in range(64):
        if p == 37:
            pairs.append((_collapsed(rng, c, 512), _collapsed(rng, c, 512)))
        else:
            d0, d1, _ = syn.make_descriptor_pair(500 + p, 128, 128)
            pairs.append((np.ascontiguousarray(d0.T), np.ascontiguousarray(d1.T)))
    sep = [q for p, q in enumerate(pairs) if p != 37]
    dists = list(_ref_dist(np.stack([a for a, _ in sep]), np.stack([b for _, b in sep]), 0))
    dists.insert(37, _ref_dist(*pairs[37], 0))
    assert (_margin(dists[37]) < EPS).mean() > 0.3
    N.profile_begin()
    res, cu0, cu1 = _run(pairs, "rows", 0.8, True, 0)
    prof = N.profile_end()
    assert prof.get("match_exact", (0.0, 0))[1] == 1 and prof.get("match_tail", (0.0, 0))[1] == 1
    _check(pairs, dists, res, cu0, cu1, 0.8, True, exact_scores=True)


@pytest.mark.gpu
def test_no_ambiguous_item_and_counter_reset():
    """A batch without any ambiguous line (empty work list) between two collapsed batches on the same workspace:
    counts and decisions of all three are right, so the work-list counters start from zero on every call."""
    coll, cdists = _reference(0)
    sep = []
    for p in range(6):
        d0, d1, _ = syn.make_descriptor_pair(700 + p, 96 + 37 * p, 80 + 41 * p)
        sep.append((np.ascontiguousarray(d0.T), np.ascontiguousarray(d1.T)))
    sdists = [np.maximum(2.0 - 2.0 * (a.astype(np.float64) @ b.T.astype(np.float64)), 0.0).astype(np.float32) for a, b in sep]
    assert all((_margin(d) >= 2 * EPS).all() and (_margin(d.T) >= 2 * EPS).all() for d in sdists)
    for pairs, dists in ((coll, cdists), (sep, sdists), (coll, cdists)):
        res, cu0, cu1 = _run(pairs, "rows", 0.8, True, 0)
        _check(pairs, dists, res, cu0, cu1, 0.8, True, exact_scores=pairs is coll)
