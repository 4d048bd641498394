"""Temperature, top-k and top-p sampling on the device: the one device rule (csrc/sample.cuh) against its fp64 host
restatement (tests/_sampling.py), token for token, in dgpt_sample and in every generation path (exact mode with the
window slide, BigramLM, the persistent decoder, the per-position CUDA graphs, the post-slide recompute), plus the
inference CLI's prompt and sampler flags."""
import numpy as np
import pytest
import torch
from scipy import stats

pytestmark = pytest.mark.gpu

import _sampling as S  # noqa: E402
from conftest import load_checkpoint, load_golden  # noqa: E402
from drakegpt_b200 import config as cfg  # noqa: E402
from drakegpt_b200 import inference, ops, train  # noqa: E402
from drakegpt_b200 import model as M  # noqa: E402
from oracle import drake_oracle as O  # noqa: E402

DEV = "cuda"
SETTINGS = [(1.0, None, 1.0), (0.8, 10, 0.9), (1.5, None, 0.5), (0.5, 40, 1.0), (1.0, 1, 1.0), (2.0, 200, 0.95),
            (0.7, None, 0.999), (1.3, 3, 0.6)]


def _settings(temperature=1.0, top_k=None, top_p=1.0):
    return ops.sampling_settings(temperature, top_k, top_p).to(DEV)


def _sample(logits, seed, step, greedy=False, sampling=None):
    out = torch.full((logits.shape[0],), -1, dtype=torch.int64, device=DEV)
    ops.raw_sample(logits, out, 0, greedy, seed, step, sampling=sampling)
    return out.cpu().numpy()


@pytest.mark.parametrize("V", [80, 300, 33, 1])
def test_sample_kernel_vs_host_restatement(V):
    """dgpt_sample_ex on seeded random logits == the fp64 rule, row for row (fp32-ambiguous rows excepted)."""
    g = torch.Generator().manual_seed(V)
    rows = 4096 if V >= 80 else 256
    logits = torch.randn(rows, V, generator=g) * 2
    logits[: rows // 8, : V // 2] = torch.round(logits[: rows // 8, : V // 2])  # exact ties, at the k-th value too
    ld = logits.to(DEV)
    host = logits.double().numpy()
    for i, (t, k, p) in enumerate(SETTINGS):
        seed, step = 1000 + 17 * i + (i << 40), 3 * i + 1
        got = _sample(ld, seed, step, sampling=_settings(t, k, p))
        frac = S.uniform(np.arange(rows), step, seed)
        skipped = 0
        for b in range(rows):
            tok, amb = S.draw(host[b], frac[b], t, k, p)
            if amb:
                skipped += 1
                continue
            assert got[b] == tok, (V, (t, k, p), b, int(got[b]), tok)
        assert skipped <= rows // 100, (V, (t, k, p), skipped)
        # greedy ignores the settings; NULL settings == the default settings, bit for bit
        assert np.array_equal(_sample(ld, seed, step, greedy=True, sampling=_settings(t, k, p)), host.argmax(1))
    assert np.array_equal(_sample(ld, 5, 9), _sample(ld, 5, 9, sampling=_settings()))


def test_filtered_distribution():
    """One row drawn 8192 x 4 times: never a removed token, frequencies match the fp64 filtered distribution."""
    g = torch.Generator().manual_seed(11)
    row = torch.randn(80, generator=g) * 1.5
    t, k, p = 0.8, 10, 0.9
    w = S.filtered(row.double().numpy(), t, k, p)
    kept = np.nonzero(w > 0)[0]
    assert 2 < len(kept) < 10
    big = row.repeat(8192, 1).to(DEV)
    counts = np.zeros(80)
    for step in range(4):
        counts += np.bincount(_sample(big, 2024, step, sampling=_settings(t, k, p)), minlength=80)
    assert counts[w == 0].sum() == 0
    expected = w[kept] / w.sum() * counts.sum()
    assert stats.chisquare(counts[kept], expected).pvalue > 1e-3


def _host_loop(kind, sd, got, t0, seed, ctx, t, k, p, logit_tol):
    """Teacher-forced host replay of generate(): for each row, the positions agree up to the first ambiguous one."""
    Bn, total = got.shape
    compared = 0
    for b in range(Bn):
        for n in range(t0, total):  # token n is drawn at step n - 1 from the prefix got[:n]
            pre = got[b:b + 1, :n] if ctx is None else got[b:b + 1, max(0, n - ctx):n]
            lg = O.forward(kind, sd, pre)[0][0, -1].double().numpy()
            tok, amb = S.draw(lg, S.uniform(np.array([b]), n - 1, seed)[0], t, k, p, logit_tol=logit_tol)
            if amb:
                break
            assert int(got[b, n]) == tok, (kind, b, n, got[b].tolist(), tok)
            compared += 1
    return compared


@pytest.mark.parametrize("kind", ["TransformerLM", "BigramLM"])
def test_generate_exact_mode_vs_host_rule(kind):
    """Shipped checkpoints (TransformerLM: fp32 mode, context 8, so the window slide is crossed)."""
    args = {"TransformerLM": (80, 32, 8, 4, 3, 0.1), "BigramLM": (80,)}[kind]
    sd = load_checkpoint(kind)
    m = getattr(M, kind)(*args)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    prompt = torch.tensor([[0, 14, 28], [1, 30, 18], [7, 7, 7]], dtype=torch.long)
    for seed in (3, 41):
        got = m.generate(prompt.to(DEV), 24, seed=seed, temperature=0.8, top_k=10, top_p=0.9).cpu()
        assert got.shape == (3, 27) and torch.equal(got[:, :3], prompt)
        n = _host_loop(kind, sd, got, 3, seed, O.context_length_of(kind, sd), 0.8, 10, 0.9, logit_tol=1e-4)
        assert n >= 0.8 * 3 * 24, n  # the exemption is the exception


@pytest.fixture(scope="module")
def scaled():
    rec = load_golden("scaled_vectors.pt")
    sd = O.synthetic_state_dict("TransformerLM", seed=rec["seed"], **rec["cfg"])
    m = M.TransformerLM(80, 384, 256, 6, 6, 0.2, precision="bf16")
    m.load_state_dict(sd)
    return m.to(DEV).eval(), sd


def _prompt(Bn, t0):
    g = torch.Generator().manual_seed(Bn * 1000 + t0)
    return torch.randint(0, 80, (Bn, t0), generator=g)


@pytest.mark.parametrize("path,Bn,t0,n_new", [("1", 3, 3, 20), ("force", 8, 3, 20), ("0", 3, 3, 20), ("1", 64, 3, 12),
                                              ("1", 2, 260, 4)])
def test_every_bf16_path(scaled, monkeypatch, path, Bn, t0, n_new):
    """Persistent decoder (3 sequences; 8 forced), per-position graphs (persistent off; batch 64), and a prompt longer
    than the 256-token window (post-slide recompute)."""
    monkeypatch.setenv("DGPT_DECODE_PERSISTENT", path)
    m, sd = scaled
    r = m.runner()
    if t0 < 256:
        assert r._persistent_decode_ok(Bn) == (path != "0" and (Bn <= 4 or path == "force"))
    prompt = _prompt(Bn, t0).to(DEV)
    greedy = m.generate(prompt, n_new, greedy=True)
    assert torch.equal(m.generate(prompt, n_new, seed=7, top_k=1, temperature=1.7), greedy)
    assert torch.equal(m.generate(prompt, n_new, seed=8, top_p=1e-6), greedy)
    a = m.generate(prompt, n_new, seed=5, top_k=5, top_p=0.95, temperature=1.2)
    assert torch.equal(a, m.generate(prompt, n_new, seed=5, top_k=5, top_p=0.95, temperature=1.2))
    assert not torch.equal(a, m.generate(prompt, n_new, seed=6, top_k=5, top_p=0.95, temperature=1.2))
    # teacher-forced on its own prefix: every token drawn with top_k=5 is in the oracle's top 5 (5th / 6th near-ties
    # excepted)
    got = m.generate(prompt, n_new, seed=9, top_k=5).cpu()
    ctx = 256
    for n in range(t0, t0 + n_new):
        lg = O.forward("TransformerLM", sd, got[:, max(0, n - ctx):n])[0][:, -1]
        top = lg.topk(6)
        ok = (top.indices[:, :5] == got[:, n:n + 1]).any(1) | ((top.values[:, 4] - top.values[:, 5]) < 5e-2)
        assert ok.all(), (n, got[:, n].tolist(), top.indices.tolist())


def test_defaults_and_graph_reuse(scaled, monkeypatch):
    """Default arguments == explicit defaults; new settings reuse the captured per-position graphs."""
    monkeypatch.setenv("DGPT_DECODE_PERSISTENT", "1")
    m, _ = scaled
    for Bn in (3, 64):
        prompt = _prompt(Bn, 2).to(DEV)
        d = m.generate(prompt, 10, seed=21)
        assert torch.equal(d, m.generate(prompt, 10, seed=21, temperature=1.0, top_k=None, top_p=1.0))
    r = m.runner()
    n_graphs = len(r.__dict__["_decode_graphs"])
    outs = [m.generate(prompt, 10, seed=21, **kw) for kw in (dict(temperature=0.5), dict(top_k=3, top_p=0.8),
                                                            dict(top_k=1))]
    assert len(r.__dict__["_decode_graphs"]) == n_graphs
    assert not torch.equal(outs[0], d) or not torch.equal(outs[1], d)
    assert torch.equal(outs[2], m.generate(prompt, 10, greedy=True))  # the buffer really is read at replay


def test_inference_cli_prompt_and_sampler(tmp_path, monkeypatch):
    train.main(["--model", "TransformerLM", "--synthetic", "6000", "--iters", "4", "--eval-interval", "2",
                "--eval-iters", "1", "--model-dir", str(tmp_path), "--generate", "0"])
    vocab = (tmp_path / "TransformerLM.pt.vocab.txt").read_text(encoding="utf-8")
    encode = inference.get_mapper(vocab)[0]
    argv = ["--model", "TransformerLM", "--length", "30", "--model-dir", str(tmp_path), "--out-dir", str(tmp_path),
            "--prompt", "ab", "--temperature", "0.7", "--top-k", "5", "--seed", "3"]
    ids, _ = inference.main(argv)
    assert ids[:2] == encode("ab") and len(ids) == 2 + 30
    assert inference.main(argv)[0] == ids
    assert inference.main(argv[:-1] + ["4"])[0] != ids
    with pytest.raises(SystemExit):
        inference.main(argv[:9] + ["a~b"])  # "~" is not in the vocabulary
    with pytest.raises(SystemExit):
        inference.main(argv + ["--top-p", "0"])
    monkeypatch.setitem(cfg.DATA, "input", str(tmp_path / "no_corpus.txt"))
    (tmp_path / "TransformerLM.pt.vocab.txt").unlink()
    with pytest.raises(SystemExit):
        inference.main(argv)  # --prompt without a vocabulary
