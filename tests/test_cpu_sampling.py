"""CPU checks of the sampling restatement (tests/_sampling.py) and of generate()'s argument validation, which runs
before any device work."""
import numpy as np
import pytest
import torch

import _sampling as S
from drakegpt_b200 import model as M
from drakegpt_b200 import ops


def test_philox_known_answers():
    """Random123's known-answer vectors for Philox4x32-10."""
    r = S.philox4x32_10((0, 0, 0, 0), (0, 0))
    assert [int(x) for x in r] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    f = 0xFFFFFFFF
    r = S.philox4x32_10((f, f, f, f), (f, f))
    assert [int(x) for x in r] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    # vectorised over rows == one row at a time
    b = np.arange(5, dtype=np.uint64)
    u = S.uniform(b, 7, (3 << 32) | 11)
    for i in range(5):
        assert u[i] == S.uniform(np.array([i], dtype=np.uint64), 7, (3 << 32) | 11)[0]
    assert np.all((u > 0) & (u < 1))


def test_top_k_keeps_ties_at_the_kth_logit():
    lg = np.array([3.0, 1.0, 2.0, 2.0, 0.5, 2.0])
    assert S.kept_set(lg, top_k=2) == {0, 2, 3, 5}  # the 2nd largest (2.0) is tied three ways: all kept
    assert S.kept_set(lg, top_k=1) == {0}
    assert S.kept_set(lg, top_k=6) == S.kept_set(lg, top_k=None) == set(range(6))


def test_filters_always_keep_the_argmax():
    g = np.random.default_rng(0)
    for _ in range(200):
        lg = g.normal(size=int(g.integers(1, 300))) * 3
        a = int(lg.argmax())
        for t, k, p in ((0.3, 1, 1.0), (1.0, None, 1e-9), (2.0, 3, 0.2), (0.7, 50, 0.95)):
            kept = S.kept_set(lg, t, k, p)
            assert a in kept
            w = S.filtered(lg, t, k, p)
            if k is not None:
                assert len(kept) <= max(k, int((lg >= np.sort(lg)[::-1][min(k, len(lg)) - 1]).sum()))
            if p < 1:  # the kept prefix is minimal: dropping its last token leaves less than top_p of the mass
                full = S.filtered(lg, t, k, 1.0)
                assert w.sum() >= p * full.sum() - 1e-12 and w.sum() - w[w > 0].min() < p * full.sum()


def test_top_k_1_and_tiny_top_p_give_the_argmax():
    g = np.random.default_rng(1)
    for _ in range(100):
        lg = g.normal(size=80) * 2
        for frac in (1e-7, 0.5, 1 - 1e-7):
            assert S.draw(lg, frac, top_k=1)[0] == int(lg.argmax())
            assert S.draw(lg, frac, temperature=3.0, top_p=1e-6)[0] == int(lg.argmax())


def test_default_rule_is_the_plain_softmax_draw():
    lg = np.array([2.0, 1.0, 0.0, -1.0, 0.5])
    p = np.exp(lg - lg.max())
    p /= p.sum()
    w = S.filtered(lg)
    assert np.allclose(w / w.sum(), p)
    cdf = np.cumsum(p)
    for frac in np.linspace(0.01, 0.99, 37):
        assert S.draw(lg, frac)[0] == int(np.searchsorted(cdf, frac, side="right"))


@pytest.mark.parametrize("kw", [dict(temperature=0), dict(temperature=-1.0), dict(temperature=float("nan")),
                                dict(temperature=float("inf")), dict(top_k=0), dict(top_k=-3), dict(top_k=2.5),
                                dict(top_p=0), dict(top_p=1.5), dict(top_p=float("nan"))])
def test_generate_rejects_bad_sampling_settings_before_the_device_check(kw):
    for m in (M.TransformerLM(80, 32, 8, 4, 3, 0.1), M.BigramLM(80)):
        with pytest.raises(ValueError):
            m.generate(torch.zeros((1, 1), dtype=torch.long), 4, **kw)


def test_sampling_settings_layout():
    t = ops.sampling_settings(0.8, 10, 0.9)
    assert t.dtype == torch.int32 and t.shape == (3,)
    f = t.view(torch.float32)
    assert f[0].item() == np.float32(0.8) and int(t[1]) == 10 and f[2].item() == np.float32(0.9)
    assert int(ops.sampling_settings()[1]) == 0  # top_k None: off
    assert int(ops.sampling_settings(top_k=10 ** 12)[1]) == 2 ** 31 - 1
    assert ops.sampling_settings(temperature=1e-60).view(torch.float32)[0].item() > 0  # 1 / temperature stays finite
