"""The tokenizer glue (linetr_b200/line_process.py) against the outputs of the reference tokenizer
(tests/golden/tokenizer_outputs.npz, written by tests/golden/make_plumbing_golden.py)."""
import types

import numpy as np
import pytest
import torch

from linetr_b200 import line_process as LP

CFGS = [{}, {"max_tokens": 8, "token_distance": 12}, {"min_length": 40, "max_keylines": 20}]


class FakeKeyLine:
    def __init__(self, x0, y0, x1, y1, octave=0):
        self.startPointX, self.startPointY, self.endPointX, self.endPointY = x0, y0, x1, y1
        self.lineLength = float(np.hypot(x1 - x0, y1 - y0)) / (2 ** octave)
        self.octave = octave


def fake_lines(seed, n, w=640, h=480):
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for _ in range(n):
        x0, y0 = rng.uniform(0, w), rng.uniform(0, h)
        ang, ln = rng.uniform(0, 2 * np.pi), rng.uniform(5, 400)
        x1, y1 = np.clip(x0 + ln * np.cos(ang), 0, w - 1), np.clip(y0 + ln * np.sin(ang), 0, h - 1)
        out.append(FakeKeyLine(float(x0), float(y0), float(x1), float(y1), int(rng.integers(0, 2))))
    out.append(FakeKeyLine(100.0, 50.0, 100.0, 300.0))   # vertical line (dx == 0 branch)
    return out


def fake_superpoint(seed, h=480, w=640):
    g = torch.Generator().manual_seed(seed)
    return {"dense_descriptor": torch.nn.functional.normalize(torch.randn(1, 256, h // 8, w // 8, generator=g), dim=1),
            "dense_score": torch.rand(1, h, w, generator=g)}


def ours(lines, sp, cfg):
    from linetr_b200.line_transformer import LineTransformer
    m = LineTransformer({"mode": "train", **cfg})
    return m.preprocess(lines, (1, 1, 480, 640), sp, None)


def test_tokenizer_shapes_and_adjacency():
    out = ours(fake_lines(3, 40), fake_superpoint(3), {})
    S = out["sublines"].shape[1]
    K = out["klines"].shape[1]
    assert out["desc_sublines"].shape == (1, S, 21, 256) and out["mask_sublines"].shape == (1, S, 22, 1)
    A = out["mat_klines2sublines"][0]
    assert A.shape == (K, S) and torch.allclose(A.sum(1), torch.ones(K))
    assert S > K  # some key lines are longer than 21 tokens * 8 px and get split


@pytest.mark.parametrize("ci", [0, 1, 2])
def test_cpu_tokenizer_glue_identical_to_reference_fixture(ci):
    """Runs everywhere (no reference checkout needed): the CPU glue against the committed outputs of the
    reference tokeniser (tests/golden/tokenizer_outputs.npz, written by make_plumbing_golden.py)."""
    from tests import helpers as H
    want = H.tokenizer_fixture(ci)
    got = ours(fake_lines(7, 60), fake_superpoint(7), CFGS[ci])
    assert set(want.keys()) | {"desc_sublines"} == set(got.keys())
    for k in want:
        assert np.array_equal(got[k].numpy(), want[k]), k
    H.check_tokenizer_desc(got["desc_sublines"].numpy(), ci)


@pytest.mark.parametrize("cfg", CFGS)
def test_tokenizer_identical_to_reference(cfg):
    """Same keys, shapes, dtypes and values as the reference tokeniser's dict."""
    from tests import helpers as H
    ci = CFGS.index(cfg)
    want = H.tokenizer_fixture(ci)
    got = ours(fake_lines(7, 60), fake_superpoint(7), cfg)
    assert set(want.keys()) | {"desc_sublines"} == set(got.keys())
    for k in want:
        assert want[k].shape == tuple(got[k].shape), k
        assert want[k].dtype == got[k].numpy().dtype, k
        assert torch.equal(torch.from_numpy(want[k]), got[k]), k
    H.check_tokenizer_desc(got["desc_sublines"].numpy(), ci)   # dtype, shape, every byte
