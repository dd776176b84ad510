"""The chained line-stage GEMM engine against the numpy oracle at production batch sizes.

`ltr_encode` runs the row-local GEMMs of the line stage and of every signature layer as one chained launch per layer
(gemm_chain2_kernel, CTA pairs over 256-row cluster tiles) when the batch has at least `chain_min_tiles()` (96) row
tiles of 128 lines and no channel-first output is asked for.  Smaller batches and `LineTransformer.forward` never take
that path, so these tests build big batches cheaply: a few distinct source pairs on the host, and on the device many
copies of them, each copy's lines reordered by its own seeded permutation.  The encoder is line-permutation-equivariant,
so every row's expected descriptor is its source image's oracle row, and every pair's expected matches are the source
pair's oracle matches, permuted.  Neighbouring tiles never hold the same content, so a misaddressed tile shows.

Every encode is counted: the number of "linear"-class launches tells which engine ran (see LINEAR_* below).

The forced_* tests run small batches with the chain forced on (LTR_CHAIN_MIN_TILES=1).  The threshold is read once per
process, so test_small_tile_counts_on_the_chain runs them in a child pytest; they skip otherwise."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from linetr_b200 import _native as N
from linetr_b200 import engine, synthetic as syn
from linetr_b200.line_transformer import LineTransformer
from oracle import linetr_oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
DESC_TOL_TIGHT = 2e-4
THRESH = 0.8

# "linear"-class launches of one ltr_encode without channel-first output (encode_impl, ltr_api.cu), 7 signature layers.
# Always: the V projection and the line position layers l4, l5 (3).
#   chained, d_inner % 256 == 0: one chain fc -> w_1 -> w_2 -> qkv_0, then per layer one chain
#       mlp1 -> mlp2 -> qkv of the next layer (the last: final projection)                        3 + 1 + 7      = 11
#   chained, d_inner % 256 != 0: fc, w_1, w_2 and qkv_0 one launch each, then the 7 layer chains      3 + 4 + 7      = 14
#   unchained: fc, w_1, w_2, per layer qkv, mlp1, mlp2, and the final projection                      3 + 3 + 21 + 1 = 28
LINEAR_CHAINED, LINEAR_CHAINED_SIG_ONLY, LINEAR_UNCHAINED = 11, 14, 28
CHAIN_MIN_TILES = 96

FORCED = os.environ.get("LTR_CHAIN_MIN_TILES") == "1"
forced_only = pytest.mark.skipif(not FORCED, reason="runs in a child process with LTR_CHAIN_MIN_TILES=1")
default_threshold = pytest.mark.skipif("LTR_CHAIN_MIN_TILES" in os.environ,
                                       reason="launch counts assume the default chain threshold")

GUARD = 256 * 1024       # bytes behind the tile image that nobody may write
SENTINEL = 0xA5

_models = {}
_oracle = {}


def model_for(tag, d_inner=1024):
    key = (tag, d_inner)
    if key not in _models:
        sd = H.standin_weights() if tag == "standin" else syn.make_state_dict(int(tag.split(":")[1]), 1, d_inner=d_inner)
        m = LineTransformer({"mode": "train", "d_inner": d_inner})
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
        _models[key] = (m.eval().to(DEV), sd)
    return _models[key]


def counted(fn):
    """-> (fn(), number of "linear"-class launches it made)."""
    N.profile_begin()
    try:
        out = fn()
    finally:
        prof = N.profile_end()
    return out, prof.get("linear", (0.0, 0))[1]


# ------------------------------------------------------------------ sources, copies, expected values
class Sources:
    """Source pairs (side 0, side 1, perm: side-1 line j is side-0 line perm[j]) and their oracle values, computed once
    per model on first use: rows [L, 256] of each side and side 0's match indices.  With `matched`, rows come from the
    oracle's match_pair (both sides at once), otherwise from one forward per image."""

    def __init__(self, key, pairs, matched=True):
        self.key, self.pairs, self.matched = key, pairs, matched

    def images(self):
        """Host images in source order: all side-0 images, then all side-1 images."""
        return [a for a, _, _ in self.pairs] + [b for _, b, _ in self.pairs]

    def n_lines(self, img):
        return int(self.images()[img]["desc_sublines"].shape[1])

    def rows(self, tag, sd, img):
        """Oracle rows of source image `img` (index into images())."""
        k = (self.key, tag, "rows", img)
        if k not in _oracle and self.matched:
            self.matches(tag, sd, img % len(self.pairs))
        if k not in _oracle:
            _oracle[k] = orc.line_transformer_forward(sd, self.images()[img])[0].T.copy()
        return _oracle[k]

    def matches(self, tag, sd, s):
        """Oracle match indices of source pair s (and both sides' rows, cached on the way)."""
        k = (self.key, tag, "match", s)
        if k not in _oracle:
            a, b, _ = self.pairs[s]
            mat, _, o0, o1 = orc.match_pair(sd, a, b, THRESH)
            _oracle[k] = orc.match_indices(mat)
            _oracle.setdefault((self.key, tag, "rows", s), o0[0].T.copy())
            _oracle.setdefault((self.key, tag, "rows", len(self.pairs) + s), o1[0].T.copy())
        return _oracle[k]


def uniform_sources(key, seeds, L, T, n_real_tokens=None, matched=True):
    return Sources(key, [syn.make_pair_inputs(s, L, T, n_real_tokens=n_real_tokens) for s in seeds], matched)


class Copies:
    """A batch made on the device: image i of the batch is source image plan[i] with its lines reordered by perms[i]
    (batch line j = source line perms[i][j])."""

    def __init__(self, src: Sources, plan, seed):
        self.src, self.plan = src, list(plan)
        rng = np.random.Generator(np.random.PCG64(seed))
        sb = engine.LineBatch.from_images(src.images()).to(DEV)
        self.perms = [rng.permutation(src.n_lines(s)) for s in self.plan]
        gather = np.concatenate([int(sb.cu_lines[s]) + p for s, p in zip(self.plan, self.perms)])
        g = torch.from_numpy(gather.astype(np.int64)).to(DEV)
        cu = np.zeros(len(self.plan) + 1, np.int32)
        cu[1:] = np.cumsum([len(p) for p in self.perms])
        self.batch = engine.LineBatch(*[t.index_select(0, g) for t in sb.tensors()], cu)
        torch.cuda.synchronize()

    @property
    def cu(self):
        return self.batch.cu_lines

    def expected_rows(self, tag, sd, i):
        return self.src.rows(tag, sd, self.plan[i])[self.perms[i]]

    def check_rows(self, tag, sd, rows, images=None):
        """rows [R, 256] (numpy) of the whole batch against the oracle, image by image; -> max |error|."""
        err = 0.0
        for i in (range(len(self.plan)) if images is None else images):
            s, e = int(self.cu[i]), int(self.cu[i + 1])
            d = float(np.abs(rows[s:e] - self.expected_rows(tag, sd, i)).max())
            assert d < DESC_TOL_TIGHT, f"image {i} (rows {s}..{e}, source {self.plan[i]}): max |desc - oracle| = {d:.3g}"
            err = max(err, d)
        return err


def packed_plan(n_src, P):
    """match_packed layout: pair p = (side 0 of source p % n_src, side 1 of the same source)."""
    return [p % n_src for p in range(P)] + [n_src + p % n_src for p in range(P)]


def expected_matches(m_src, perm0, perm1):
    """Source match m_src (side-0 line x -> side-1 line m_src[x] or -1) seen through the copies' permutations:
    copy line i is source line perm0[i], so it matches the copy's side-1 line j with perm1[j] == m_src[perm0[i]]."""
    inv1 = np.argsort(perm1)
    m = m_src[perm0]
    return np.where(m >= 0, inv1[np.maximum(m, 0)], -1).astype(np.int32)


def check_pair_matches(res, tag, sd, src, side0: Copies, i0, side1: Copies, i1, p):
    s = side0.plan[i0]
    want = expected_matches(src.matches(tag, sd, s), side0.perms[i0], side1.perms[i1])
    got = res.pair(p).cpu().numpy()
    assert np.array_equal(got, want), f"pair {p}: {(got != want).sum()} of {len(want)} matches differ from the oracle"
    assert int(res.counts[p]) == int((want >= 0).sum()), f"pair {p}: count"


# ------------------------------------------------------------------ C ABI encode into a guarded tile image
def sw128_offset(row, k):
    """Byte offset of element (row, k) inside a 128 x 64 bf16 K-major SWIZZLE_128B tile (ptx_sm100.cuh:362)."""
    return (row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 3) ^ (row & 7)) & 7) << 4) + (k & 7) * 2


def decode_tiles(img, R):
    """The descriptor tile image of ltr_encode (tiles_image, ltr_api.cu) -> (hi, lo) bf16 bit patterns [R, 256].
    A hi plane, then a lo plane, of align_up(R, 128) * 256 bf16 each; in a plane, tile (mt * 4 + kb) of 128 x 64
    elements holds rows mt*128.. and columns kb*64.., element (r, k) at byte sw128_offset(r, k) of the tile."""
    u16 = img.view(np.uint16)
    plane = -(-R // 128) * 128 * 256
    assert u16.size == 2 * plane
    r = np.arange(R, dtype=np.int64)[:, None]
    k = np.arange(256, dtype=np.int64)[None, :]
    off = ((r >> 7) * 4 + (k >> 6)) * (128 * 64) + sw128_offset(r & 127, k & 63) // 2
    return u16[off], u16[plane + off]


def bf16_rn(x):
    """fp32 -> bf16 bit pattern, round to nearest even (finite inputs)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def bf16_f32(h):
    return (h.astype(np.uint32) << 16).view(np.float32)


def encode_guarded(model, batch: engine.LineBatch):
    """ltr_encode through the C ABI with rows and the tile image on, the tile buffer followed by a GUARD-byte band and
    all of it pre-filled with SENTINEL.  -> (rows [R, 256], tile image bytes, guard band bytes, linear launches)."""
    h = model._get_handle(DEV)
    lib = N.load()
    R, T = batch.n_lines, batch.n_tokens
    nbytes = int(lib.ltr_desc_tiles_bytes(R))
    buf = torch.full((nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device=DEV)
    rows = torch.empty((R, 256), dtype=torch.float32, device=DEV)
    ws = h.workspace(batch.n_images, R, T)
    L = batch.uniform_lines
    cu = np.ascontiguousarray(batch.cu_lines, dtype=np.int32)
    cu_dev = batch.dev_i32("cu_lines", DEV)
    ragged = L is None
    w, hgt = model._image_wh()
    inp = N.LtrEncodeInput(*[t.data_ptr() for t in batch.tensors()], cu.ctypes.data if ragged else None,
                           cu_dev.data_ptr() if ragged else None, batch.n_images, R, T, 0 if ragged else L,
                           float(w), float(hgt))
    outp = N.LtrEncodeOutput(None, rows.data_ptr(), buf.data_ptr())

    def run():
        with torch.cuda.device(DEV):
            rc = lib.ltr_encode(h.ptr, C.byref(inp), C.byref(outp), C.c_void_p(ws.data_ptr()), ws.numel(),
                                C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream))
        N.check(rc, "ltr_encode")
    _, n_lin = counted(run)
    b = buf.cpu().numpy()
    return rows.cpu().numpy(), b[:nbytes], b[nbytes:], n_lin


def check_tile_image(rows, img, guard):
    """Nothing written behind the image; the image holds every row split into bf16 hi + lo."""
    bad = np.nonzero(guard != SENTINEL)[0]
    assert bad.size == 0, f"{bad.size} bytes written past the tile image (first at +{bad[0] if bad.size else 0})"
    hi, lo = decode_tiles(img, rows.shape[0])
    # both chain epilogues (streamed, gemm_chain2_kernel; staged, epi_store_image) store the fp32 row and split the same
    # registers (split8_bf16, ptx_sm100.cuh:392, bit-identical to split_bf16: hi = bf16_rn(x), lo = bf16_rn(x - hi))
    want_hi = bf16_rn(rows)
    want_lo = bf16_rn(rows - bf16_f32(want_hi))
    bad_rows = np.nonzero((hi != want_hi).any(1) | (lo != want_lo).any(1))[0]
    assert bad_rows.size == 0, f"{bad_rows.size} rows of the tile image differ from the fp32 rows (first: {bad_rows[:8]})"


# ------------------------------------------------------------------ 1. cfg1 at bench size
@default_threshold
@pytest.mark.parametrize("tag", ["standin", "synthetic:0:1"])
def test_cfg1_bench_size_chained(tag):
    """64 pairs x 128 lines x 21 tokens through match_packed: 128 row tiles, the encoder writes the matcher's tile image."""
    model, sd = model_for(tag)
    src = uniform_sources("cfg1", (1000, 1001, 1002), 128, 21)
    P = 64
    cp = Copies(src, packed_plan(3, P), seed=1)
    eng = engine.PairEngine(model, DEV)
    res, n_lin = counted(lambda: eng.match_packed(cp.batch, P, THRESH, keep_desc=True))
    assert n_lin == LINEAR_CHAINED
    rows = torch.cat([res.desc0, res.desc1]).cpu().numpy()
    assert np.abs(np.linalg.norm(rows, axis=1) - 1).max() < 1e-5
    cp.check_rows(tag, sd, rows)
    for p in range(P):
        check_pair_matches(res, tag, sd, src, cp, p, cp, P + p, p)


# ------------------------------------------------------------------ 2. cfg2 shape
@default_threshold
def test_cfg2_shape_chained():
    """48 pairs x 256 lines x 32 tokens (192 row tiles), match_packed with the tile image."""
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src = uniform_sources("cfg2", (2000, 2001), 256, 32)
    P = 48
    cp = Copies(src, packed_plan(2, P), seed=2)
    eng = engine.PairEngine(model, DEV)
    res, n_lin = counted(lambda: eng.match_packed(cp.batch, P, THRESH, keep_desc=True))
    assert n_lin == LINEAR_CHAINED
    rows = torch.cat([res.desc0, res.desc1]).cpu().numpy()
    assert np.abs(np.linalg.norm(rows, axis=1) - 1).max() < 1e-5
    cp.check_rows(tag, sd, rows)
    for p in range(P):
        check_pair_matches(res, tag, sd, src, cp, p, cp, P + p, p)


# ------------------------------------------------------------------ 3. odd tile count with a tile image
@default_threshold
def test_odd_tile_count_tile_image_stays_inside():
    """97 images x 128 lines: the last cluster of CTA pairs has one real tile.  The tile image is exactly
    ltr_desc_tiles_bytes(R) long; the encoder must not write behind it nor over its first rows, and every row's
    tiles must be the bf16 split of the row.  Only then match_pairs (both sides 97 tiles, real allocations)."""
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src = uniform_sources("odd97", (3000, 3001), 128, 21)
    P = 97
    side0 = Copies(src, [p % 2 for p in range(P)], seed=3)
    assert -(-side0.batch.n_lines // 128) == P
    rows, img, guard, n_lin = encode_guarded(model, side0.batch)
    assert n_lin == LINEAR_CHAINED
    check_tile_image(rows, img, guard)
    side0.check_rows(tag, sd, rows)

    side1 = Copies(src, [2 + p % 2 for p in range(P)], seed=4)
    eng = engine.PairEngine(model, DEV)
    res, n_lin = counted(lambda: eng.match_pairs(side0.batch, side1.batch, THRESH, keep_desc=True))
    assert n_lin == 2 * LINEAR_CHAINED
    side1.check_rows(tag, sd, res.desc1.cpu().numpy())
    for p in range(P):
        check_pair_matches(res, tag, sd, src, side0, p, side1, p, p)


# ------------------------------------------------------------------ 4. ragged at scale
def ragged_sources(R_side0):
    """cfg3-class source pairs (64 token slots, 5..64 real tokens) of 32, 512, 91, 300 and 437 lines plus two fillers,
    and the side-0 plan of a batch whose copies sum to exactly R_side0 lines.  The plan ends with a filler, the 91- and
    the 32-line image, so that near the end of the whole batch (side 1 mirrors side 0) the last image lies inside the
    partial last tile and two other images straddle the boundaries of the last two cluster tiles."""
    Ls = [32, 512, 91, 300, 437]
    tail = Ls[2] + Ls[0]
    plan, s = [], 0
    while R_side0 - tail - s > 1024:
        plan.append(len(plan) % len(Ls))
        s += Ls[plan[-1]]
    rest = R_side0 - tail - s               # in (512, 1024]: two fillers of 257..512 lines
    Ls += [rest // 2, rest - rest // 2]
    plan += [len(Ls) - 2, len(Ls) - 1, 2, 0]
    pairs = [syn.make_pair_inputs(4000 + i, L, 64, n_real_tokens=(5, 64)) for i, L in enumerate(Ls)]
    return Sources(("ragged", R_side0), pairs, matched=False), plan


@default_threshold
def test_cfg3_ragged_odd_tiles_chained():
    """Ragged 32..512-line images, R % 128 != 0 and an odd number (97) of row tiles, through match_packed.  Against the
    oracle: the smallest and the largest image (L > 128: the attention kernel's multi-tile path), the images that
    straddle the boundaries of the last two cluster tiles (256 rows each) and the image ending in the partial last tile
    (with every other copy of the same source images).  Every pair's matches recover its known permutation."""
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src, plan0 = ragged_sources(6170)
    n_src = len(src.pairs)
    P = len(plan0)
    cp = Copies(src, plan0 + [n_src + s for s in plan0], seed=5)
    R = cp.batch.n_lines
    tiles = -(-R // 128)
    assert R % 128 != 0 and tiles % 2 == 1 and tiles >= CHAIN_MIN_TILES
    eng = engine.PairEngine(model, DEV)
    res, n_lin = counted(lambda: eng.match_packed(cp.batch, P, THRESH, keep_desc=True))
    assert n_lin == LINEAR_CHAINED
    rows = torch.cat([res.desc0, res.desc1]).cpu().numpy()
    assert np.abs(np.linalg.norm(rows, axis=1) - 1).max() < 1e-5

    cu = cp.cu
    sizes = np.diff(cu)
    n_ct = (tiles + 1) // 2
    last = len(sizes) - 1
    assert cu[last] > 128 * (tiles - 1)              # the last image lies inside the partial last tile
    picks = {int(np.argmin(sizes)), int(np.argmax(sizes)), last}
    for bnd in (256 * (n_ct - 2), 256 * (n_ct - 1)):
        straddle = np.nonzero((cu[:-1] < bnd) & (cu[1:] > bnd))[0]
        assert straddle.size == 1 and straddle[0] not in picks, f"row {bnd}: pick other lengths"
        picks.add(int(straddle[0]))
    assert sizes.min() == 32 and sizes.max() == 512 and len(picks) == 5
    want_src = {cp.plan[i] for i in picks}
    cp.check_rows(tag, sd, rows, images=[i for i in range(len(cp.plan)) if cp.plan[i] in want_src])

    for p in range(P):
        perm = src.pairs[plan0[p]][2]
        p0, p1 = cp.perms[p], cp.perms[P + p]
        m = res.pair(p).cpu().numpy()
        ok = m >= 0
        assert ok.sum() >= 0.9 * len(m), f"pair {p}: {ok.sum()} of {len(m)} lines matched"
        assert np.array_equal(perm[p1[m[ok]]], p0[ok]), f"pair {p}: wrong matches"
        assert int(res.counts[p]) == int(ok.sum())


# ------------------------------------------------------------------ 5. FFN widths
@default_threshold
@pytest.mark.parametrize("d_inner,want_linear", [(512, LINEAR_CHAINED), (384, LINEAR_CHAINED_SIG_ONLY)])
def test_ffn_width_on_chained_path(d_inner, want_linear):
    """d_inner = 512 runs the line stage on the chain too; 384 is not a multiple of 256, so only the signature layers
    chain.  97 images x 128 lines."""
    tag = "synthetic:3"
    model, sd = model_for(tag, d_inner)
    src = uniform_sources(("ffn", d_inner), (5000, 5001), 128, 21, n_real_tokens=(3, 21), matched=False)
    cp = Copies(src, [i % 2 for i in range(97)], seed=6)
    eng = engine.PairEngine(model, DEV)
    rows, n_lin = counted(lambda: eng.encode(cp.batch))
    assert n_lin == want_linear
    cp.check_rows((tag, d_inner), sd, rows.cpu().numpy())


# ------------------------------------------------------------------ 6. chained vs unchained
@default_threshold
def test_chained_equals_unchained():
    """The cfg1 batch of test_cfg1_bench_size_chained encoded whole (128 tiles: chained) and as two halves of 64 tiles
    (unchained); the same rows to within the descriptor tolerance."""
    model, _ = model_for("synthetic:0:1")
    src = uniform_sources("cfg1", (1000, 1001, 1002), 128, 21)
    cp = Copies(src, packed_plan(3, 64), seed=1)
    eng = engine.PairEngine(model, DEV)
    whole, n_lin = counted(lambda: eng.encode(cp.batch))
    assert n_lin == LINEAR_CHAINED
    b = cp.batch
    half = b.n_lines // 2
    parts = []
    for s in (slice(0, half), slice(half, None)):
        hb = engine.LineBatch(*[t[s] for t in b.tensors()], np.arange(65, dtype=np.int32) * 128)
        r, n_lin = counted(lambda: eng.encode(hb))
        assert n_lin == LINEAR_UNCHAINED
        parts.append(r)
    diff = float((whole - torch.cat(parts)).abs().max())
    print(f"max |chained - unchained| = {diff:.3e}")
    assert diff < DESC_TOL_TIGHT


# ------------------------------------------------------------------ 7. small tile counts with the chain forced
@pytest.mark.skipif(FORCED, reason="parent of the forced_* tests")
def test_small_tile_counts_on_the_chain():
    """The forced_* tests in a child pytest with LTR_CHAIN_MIN_TILES=1: tile counts (1, 2, 3, 5, ragged, 64-line images)
    that no default batch size runs on the chain."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, LTR_CHAIN_MIN_TILES="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", os.path.join("tests", "test_chain_parity.py"), "-m", "gpu", "-k", "forced",
        "-p", "no:cacheprovider", "-q"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root, env=env)
    log = out.stdout[-6000:] + out.stderr[-3000:]
    assert out.returncode == 0, log
    passed = re.search(r"(\d+) passed", out.stdout)
    assert passed and int(passed.group(1)) == N_FORCED and "skipped" not in out.stdout.splitlines()[-1], log


N_FORCED = 6   # forced_* test cases below


def _forced_check(tag, sd, model, cp):
    rows, img, guard, n_lin = encode_guarded(model, cp.batch)
    assert n_lin == LINEAR_CHAINED
    check_tile_image(rows, img, guard)
    cp.check_rows(tag, sd, rows)


@forced_only
@pytest.mark.parametrize("n_tiles", [1, 2, 3, 5])
def test_forced_uniform_tiles(n_tiles):
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src = uniform_sources("forced128", (6000, 6001), 128, 21, n_real_tokens=(3, 21), matched=False)
    _forced_check(tag, sd, model, Copies(src, [i % 2 for i in range(n_tiles)], seed=7 + n_tiles))


@forced_only
def test_forced_ragged_300_lines():
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src = Sources("forced300", [syn.make_pair_inputs(6100 + i, L, 32, n_real_tokens=(2, 32))
                                for i, L in enumerate((37, 140, 123))], matched=False)
    cp = Copies(src, [0, 1, 2], seed=20)
    assert cp.batch.n_lines == 300 and cp.batch.uniform_lines is None
    _forced_check(tag, sd, model, cp)


@forced_only
def test_forced_64_line_images():
    tag = "synthetic:0:1"
    model, sd = model_for(tag)
    src = uniform_sources("forced64", (6200, 6201), 64, 21, matched=False)
    _forced_check(tag, sd, model, Copies(src, [0, 1, 2, 3, 0], seed=21))
