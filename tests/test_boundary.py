"""CPU-only checks of the drop-in boundary: module surface, state-dict contract, C-ABI
exports, host-side glue.  No compute call is made (there is no GPU here and no fallback)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from linetr_b200 import _native as N
from linetr_b200 import synthetic as syn
from linetr_b200.line_transformer import LineTransformer
from linetr_b200 import nn_matcher as nnm
from linetr_b200 import engine
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(nd=1):
    return LineTransformer({"mode": "train", "n_line_descriptive_layers": nd})


def test_header_symbols_exported():
    hdr = open(os.path.join(ROOT, "include", "linetr_b200.h")).read()
    declared = set(re.findall(r"\b(ltr_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(N.EXPORTED_SYMBOLS), declared ^ set(N.EXPORTED_SYMBOLS)
    lib = ctypes.CDLL(N.lib_path())
    for s in declared:
        assert hasattr(lib, s), f"{s} not exported"
    dbg = open(os.path.join(ROOT, "include", "linetr_b200_debug.h")).read()
    declared_dbg = set(re.findall(r"\b(ltr_[a-z_0-9]+)\s*\(", dbg))
    assert declared_dbg == set(N.DEBUG_SYMBOLS)
    for s in declared_dbg:
        assert hasattr(lib, s), f"{s} not exported"
    assert N.load().ltr_abi_version() == N.ABI_VERSION == 3


def test_header_constants_match_binding_and_kernels():
    """The constants the C header, the ctypes binding and the kernels each spell out must agree (the exchange buffer of
    the multi-GPU count publication is sized and indexed by LTR_GATHER_SLOTS on all three sides)."""
    hdr = open(os.path.join(ROOT, "include", "linetr_b200.h")).read()
    slots = int(re.search(r"#define\s+LTR_GATHER_SLOTS\s+(\d+)", hdr).group(1))
    abi = int(re.search(r"#define\s+LTR_ABI_VERSION\s+(\d+)", hdr).group(1))
    cu = open(os.path.join(ROOT, "linetr_b200", "csrc", "match_tc.cuh")).read()
    assert slots == N.GATHER_SLOTS == int(re.search(r"constexpr int GATHER_SLOTS = (\d+);", cu).group(1))
    assert abi == N.ABI_VERSION
    assert slots >= 6   # one exchange may stay in flight across a step boundary (DESIGN.md section 6)


def test_state_dict_contract():
    m = _model()
    spec = syn.state_dict_spec(1)
    sd = m.state_dict()
    assert list(sd.keys()) == [k for k, _, _ in spec]
    assert len(sd) == 198
    for k, shape, _ in spec:
        assert tuple(sd[k].shape) == tuple(shape), k
    m.load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(3, 1).items()}, strict=True)
    with pytest.raises(RuntimeError):
        _model(4).load_state_dict({k: torch.from_numpy(v) for k, v in syn.make_state_dict(3, 1).items()})


def test_shipped_checkpoint_loads_strict(tmp_path):
    with open(os.path.join(H.GOLDEN_DIR, "checkpoint_stats.json")) as f:
        shipped_keys = list(json.load(f))            # the shipped checkpoint's keys, in its order
    p = H.save_standin_checkpoint(tmp_path / "LineTR_weight.pth")
    m = LineTransformer({"mode": "test", "weights_path": p})
    ref = torch.load(p, map_location="cpu")
    assert list(ref.keys()) == shipped_keys
    assert list(m.state_dict().keys()) == shipped_keys
    for k, v in ref.items():
        assert torch.equal(m.state_dict()[k], v), k


def test_same_keys_and_init_as_reference():
    """Against the reference's random init (tests/golden/reference_init.json): same keys in the same order,
    shapes, dtypes and - same RNG consumption - the same values; same config."""
    with open(os.path.join(H.GOLDEN_DIR, "reference_init.json")) as f:
        want = json.load(f)
    torch.manual_seed(0)
    o = _model(2)
    sd = o.state_dict()
    assert list(sd.keys()) == [t["key"] for t in want["tensors"]]
    for t in want["tensors"]:
        v = sd[t["key"]]
        assert list(v.shape) == t["shape"] and str(v.dtype) == t["dtype"], t["key"]
        flat = v.reshape(-1).double().numpy()
        assert flat.sum() == t["sum"], t["key"]
        assert flat[t["idx"]].tolist() == t["values"], t["key"]
    assert o.config == want["config"]


def test_config_and_defaults():
    m = LineTransformer({"mode": "train", "nn_threshold": 0.8, "max_tokens": 32})
    assert m.config["nn_threshold"] == 0.8 and m.config["max_tokens"] == 32 and m.config["min_length"] == 16
    m.config["min_length"] = 20  # Matching mutates it (models/matching.py:31)
    d = m.default_ret()
    assert tuple(d["line_desc"].shape) == (1, 256, 0) and tuple(d["klines"].shape) == (1, 0, 2, 2)
    assert tuple(d["mat_klines2sublines"].shape) == (1, 0, 0)
    out = m({"klines": []})
    assert tuple(out["line_desc"].shape) == (1, 256, 0)


def test_no_cpu_fallback():
    m = _model()
    data = {k: torch.from_numpy(v) for k, v in syn.make_image_inputs(1, 4, 21).items()}
    with pytest.raises(N.LtrError):
        m(data)
    if not torch.cuda.is_available():
        with pytest.raises(N.LtrError):
            nnm.nn_matcher_distmat(np.zeros((1, 3, 3), np.float32), 0.8)


def test_matcher_empty_inputs():
    assert nnm.nn_matcher_distmat(np.zeros((1, 0, 5), np.float32), 0.8).shape == (1, 0, 5)
    mat, dist = nnm.nn_matcher(np.zeros((256, 0), np.float32), np.zeros((256, 7), np.float32))
    assert mat.shape == (1, 0, 7) and dist.shape == (1, 0, 7) and mat.dtype == np.float64


def test_adjacency_to_csr():
    A = np.zeros((3, 6), np.float32)
    A[0, 0:1] = 1
    A[1, 1:4] = 1 / 3
    A[2, 4:6] = 0.5
    assert nnm.adjacency_to_csr(A).tolist() == [0, 1, 4, 6]
    A[1, 1] = 0.5
    with pytest.raises(N.LtrError):
        nnm.adjacency_to_csr(A)


def test_linebatch_layouts():
    ims = [syn.make_image_inputs(s, L, 21) for s, L in ((1, 5), (2, 9), (3, 1))]
    b = engine.LineBatch.from_images(ims)
    assert b.cu_lines.tolist() == [0, 5, 14, 15] and b.n_lines == 15 and b.uniform_lines is None
    assert tuple(b.desc.shape) == (15, 21, 256) and b.sub_off is None
    st = engine.LineBatch.from_stacked(H.stack([syn.make_image_inputs(s, 6, 21) for s in (4, 5)]))
    assert st.uniform_lines == 6 and st.n_images == 2
    assert torch.equal(st.desc[6:], torch.from_numpy(syn.make_image_inputs(5, 6, 21)["desc_sublines"][0]))


def test_shard_range_partitions():
    for n in (0, 1, 7, 64, 513):
        for w in (1, 2, 4, 8):
            spans = [engine.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [e - s for s, e in spans]
            assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n_total = 11
    s, e = engine.shard_range(n_total, rank, world)
    local = torch.arange(s, e, dtype=torch.int32) * 3 + 1
    got = engine.gather_counts(local, n_total)
    q.put((rank, got.tolist()))
    dist.destroy_process_group()


def test_gather_counts_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    want = (np.arange(11) * 3 + 1).tolist()
    assert res[0] == want and res[1] == want
