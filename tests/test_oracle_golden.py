"""Pin the CPU oracle (oracle/drake_oracle.py) to outputs of the real reference.

Every fixture here was produced by tests/golden/make_golden.py from the
unmodified reference code; the oracle must reproduce them (fp32 CPU, same torch
ops -> tolerances are at rounding level).
"""
import torch
import pytest

from oracle import drake_oracle as O
from conftest import load_golden, load_checkpoint

# train_curves.pt was recorded with 8 CPU threads.  The summation order of torch's CPU kernels depends on the thread
# count, and 200 steps of the TransformerLM curve amplify a last-bit difference at step 3 to 1e-3 by the end.
CURVE_THREADS = 8


@pytest.fixture
def curve_threads():
    before = torch.get_num_threads()
    torch.set_num_threads(CURVE_THREADS)
    yield
    torch.set_num_threads(before)


@pytest.mark.parametrize("kind", O.KINDS)
def test_checkpoint_logits_loss_greedy(kind):
    rec = load_golden("ckpt_vectors.pt")[kind]
    sd = load_checkpoint(kind)
    cfg = O.infer_config(kind, sd)
    schema = O.state_dict_schema(kind, **{**dict(head_size=32), **cfg}) if kind != "BigramLM" else \
        O.state_dict_schema(kind, cfg["vocab_size"])
    assert list(schema.keys()) == list(sd.keys())
    assert all(tuple(sd[k].shape) == tuple(s) for k, s in schema.items())
    for case in rec["cases"]:
        lg, _ = O.forward(kind, sd, case["idx"])
        assert lg.shape == case["logits"].shape
        torch.testing.assert_close(lg, case["logits"], rtol=1e-5, atol=1e-5)
        lg2, loss = O.forward(kind, sd, case["idx"], case["targets"])
        assert lg2.shape == (case["idx"].numel(), lg.shape[-1])
        torch.testing.assert_close(loss, case["loss"], rtol=1e-6, atol=1e-6)
    g1 = O.generate(kind, sd, torch.zeros((1, 1), dtype=torch.long), 64, greedy=True)
    assert torch.equal(g1, rec["greedy_1"])
    g3 = O.generate(kind, sd, torch.tensor([[0], [14], [30]]), 40, greedy=True)
    assert torch.equal(g3, rec["greedy_3"])


@pytest.mark.parametrize("kind", O.KINDS)
def test_checkpoint_grads(kind):
    rec = load_golden("ckpt_vectors.pt")[kind]
    sd = load_checkpoint(kind)
    case = rec["cases"][3]
    _, _, grads = O.loss_and_grads(kind, sd, case["idx"], case["targets"], dropout=0.0, training=False)
    for k, g in rec["grads"].items():
        if g is None:
            assert grads[k] is None  # ln_f never receives a gradient (SURVEY Q1)
        else:
            torch.testing.assert_close(grads[k], g, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("key,kind,p", [
    ("BigramLM", "BigramLM", 0.0), ("SingleHeadAttentionLM", "SingleHeadAttentionLM", 0.0),
    ("MultiHeadAttentionLM", "MultiHeadAttentionLM", 0.0), ("BlocksLM", "BlocksLM", 0.0),
    ("ResidualBlocksLM", "ResidualBlocksLM", 0.0), ("TransformerLM", "TransformerLM", 0.0),
    ("TransformerLM_p0.1", "TransformerLM", 0.1)])
def test_train_curve_200_steps(key, kind, p, curve_threads):
    gold = load_golden("train_curves.pt")
    g = torch.Generator().manual_seed(gold["batches_seed"])
    batches = [(torch.randint(0, 80, (32, 8), generator=g), torch.randint(0, 80, (32, 8), generator=g))
               for _ in range(200)]
    sd = load_checkpoint(kind)
    torch.manual_seed(4242)  # same dropout stream as the reference run
    losses = O.train_steps(kind, sd, batches, lr=1e-3, dropout=p, training=True)
    ref = gold[key]["losses"]
    rel = (torch.tensor(losses, dtype=torch.float64) - ref).abs() / ref
    assert rel.max() < 2e-4, rel.max()
    fin = sd.get("lm_head.weight", sd["token_embedding_table.weight"])
    torch.testing.assert_close(fin, gold[key]["final_lm_or_tok"], rtol=1e-3, atol=1e-4)
    if gold[key]["final_ln_f"] is not None:
        assert torch.equal(sd["ln_f.weight"], gold[key]["final_ln_f"])  # untouched, exactly 1


def test_scaled_shape():
    rec = load_golden("scaled_vectors.pt")
    sd = O.synthetic_state_dict("TransformerLM", seed=rec["seed"], **rec["cfg"])
    assert sum(v.numel() for k, v in sd.items() if not k.endswith("tril")) == rec["n_params"] == 10800464
    lg, loss, grads = O.loss_and_grads("TransformerLM", sd, rec["idx"], rec["targets"], training=False)
    torch.testing.assert_close(loss, rec["loss"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(lg[:: rec["row_stride"]], rec["logits_rows"], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(grads["lm_head.weight"], rec["grad_lm_head"], rtol=1e-3, atol=1e-6)
    torch.testing.assert_close(grads["blocks.0.sa_head.heads.0.key.weight"], rec["grad_qkv_l0h0_key"], rtol=1e-3, atol=1e-6)
    torch.testing.assert_close(grads["position_embedding_table.weight"], rec["grad_pos"], rtol=1e-3, atol=1e-6)
    g1 = O.generate("TransformerLM", sd, torch.zeros((1, 1), dtype=torch.long), 24, greedy=True)
    assert torch.equal(g1, rec["greedy_1"])


def test_misc():
    m = load_golden("misc_vectors.pt")
    enc, dec, vs = O.get_mapper(m["tok"]["text"])
    assert vs == m["tok"]["vocab_size"]
    assert enc(m["tok"]["probe"]) == m["tok"]["ids"]
    assert enc(m["tok"]["text"]) == m["tok"]["all_ids"]
    assert dec(m["tok"]["all_ids"]) == m["tok"]["text"]
    torch.manual_seed(m["get_batch"]["seed"])
    data = torch.arange(1000, dtype=torch.long) % 80
    x, y = O.get_batch(data, 8, 4)
    assert torch.equal(x, m["get_batch"]["x"]) and torch.equal(y, m["get_batch"]["y"])
    P = dict(context_length=8, embedding_dim=32, num_layers=3)
    S = dict(context_length=256, embedding_dim=384, num_layers=6)
    for (k, s), v in m["model_params"].items():
        assert O.model_params(S if s else P, k, 80) == v
    for i, lr in enumerate(m["cyclic_lr"]):
        assert abs(O.cyclic_lr(i, 1e-3, 5e-3) - lr) < 1e-12
    a = m["adamw"]
    sd = {"a": a["a0"].clone(), "b": a["b0"].clone()}
    opt = O.AdamW(sd, a["lr"])
    for g in a["grads"]:
        opt.step({"a": g, "b": None})
    torch.testing.assert_close(sd["a"], a["a3"], rtol=1e-6, atol=1e-7)
    assert torch.equal(sd["b"], a["b3"])
    for k, n in m["param_counts"].items():
        sdk = load_checkpoint(k)
        assert sum(v.numel() for kk, v in sdk.items() if not kk.endswith("tril")) == n
