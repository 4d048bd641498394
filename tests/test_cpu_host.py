"""CPU-only checks: library builds/loads and exports the whole C-ABI, host-side logic
(state_dict layout, tokenizer, config, bucket planning, loud failure without a GPU)."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT, load_checkpoint, load_golden
from oracle import drake_oracle as O

CFG = {"BigramLM": (80,), "SingleHeadAttentionLM": (80, 32, 8, 32), "MultiHeadAttentionLM": (80, 32, 8, 32, 4),
       "BlocksLM": (80, 32, 8, 4, 3), "ResidualBlocksLM": (80, 32, 8, 4, 3), "TransformerLM": (80, 32, 8, 4, 3, 0.1)}


def test_library_exports_every_declared_symbol():
    from drakegpt_b200 import _lib, build
    lib = build.build()
    handle = ctypes.CDLL(lib)
    header = open(os.path.join(ROOT, "include", "drakegpt_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(dgpt_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    for sym in declared:
        assert hasattr(handle, sym), f"{sym} declared in include/drakegpt_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == declared
    assert handle.dgpt_abi_version() == 2
    # host-side helper works without a GPU and is deterministic
    handle.dgpt_dropout_keep_host.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_float]
    keeps = [handle.dgpt_dropout_keep_host(42, 1, i, 0.2) for i in range(20000)]
    assert 0.78 < sum(keeps) / len(keeps) < 0.82
    assert keeps == [handle.dgpt_dropout_keep_host(42, 1, i, 0.2) for i in range(20000)]
    assert keeps != [handle.dgpt_dropout_keep_host(43, 1, i, 0.2) for i in range(20000)]


def test_compute_entry_points_fail_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from drakegpt_b200 import _lib
    assert _lib.lib().dgpt_device_check() != 0
    with pytest.raises(_lib.KernelError):
        _lib.require_gpu()
    from drakegpt_b200 import model as M
    with pytest.raises(_lib.KernelError):
        M.BigramLM(80)(torch.zeros((1, 4), dtype=torch.long))
    with pytest.raises(_lib.KernelError):
        M.TransformerLM(80, 32, 8, 4, 3, 0.1).generate(torch.zeros((1, 1), dtype=torch.long), 4)


@pytest.mark.parametrize("kind", O.KINDS)
def test_state_dict_layout_matches_reference_checkpoints(kind):
    from drakegpt_b200 import model as M
    sd = load_checkpoint(kind)
    m = getattr(M, kind)(*CFG[kind])
    fresh = m.state_dict()
    assert list(fresh.keys()) == list(sd.keys())
    assert all(fresh[k].shape == sd[k].shape and fresh[k].dtype == sd[k].dtype for k in sd)
    res = m.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    out = m.state_dict()
    assert all(torch.equal(out[k], sd[k]) for k in sd)
    n_params = sum(p.numel() for p in m.parameters())
    assert n_params == load_golden("misc_vectors.pt")["param_counts"][kind]
    bad = dict(sd)
    bad.pop(next(k for k in sd if k.endswith("weight")))
    with pytest.raises(RuntimeError):
        getattr(M, kind)(*CFG[kind]).load_state_dict(bad, strict=True)
    if kind != "BigramLM":
        worse = dict(sd)
        key = next(k for k in sd if k.endswith("tril"))
        worse[key] = torch.ones_like(sd[key])  # not causal
        with pytest.raises(RuntimeError):
            getattr(M, kind)(*CFG[kind]).load_state_dict(worse, strict=True)


def test_scaled_model_shape_and_precision_choice():
    from drakegpt_b200 import model as M
    m = M.TransformerLM(80, 384, 256, 6, 6, 0.2)
    assert m.precision == "bf16" and M.count_parameters(m) == 10800464 and len(m.state_dict()) == 210
    assert M.TransformerLM(80, 32, 8, 4, 3, 0.1).precision == "fp32"
    gold = load_golden("misc_vectors.pt")
    P = dict(context_length=8, embedding_dim=32, num_layers=3)
    S = dict(context_length=256, embedding_dim=384, num_layers=6)
    for (k, s), v in gold["model_params"].items():
        assert M.model_params(S if s else P, k, 80) == v
    assert m.blocks[0].sa_head.heads[5].key.weight.shape == (64, 384)
    from drakegpt_b200.model_component import Head, SingleHeadAttention
    assert SingleHeadAttention is Head


def test_tokenizer_config_and_batcher():
    from drakegpt_b200 import config, preprocessing
    gold = load_golden("misc_vectors.pt")
    enc, dec, vs = preprocessing.get_mapper(gold["tok"]["text"])
    assert vs == gold["tok"]["vocab_size"]
    assert enc(gold["tok"]["probe"]) == gold["tok"]["ids"] and enc(gold["tok"]["text"]) == gold["tok"]["all_ids"]
    assert dec(gold["tok"]["all_ids"]) == gold["tok"]["text"]
    with pytest.raises(KeyError):
        enc("☃")
    torch.manual_seed(gold["get_batch"]["seed"])
    data = torch.arange(1000, dtype=torch.long) % 80
    x, y = preprocessing.get_batch(data, 8, 4, torch.device("cpu"))
    assert torch.equal(x, gold["get_batch"]["x"]) and torch.equal(y, gold["get_batch"]["y"])
    assert config.PARAMS["context_length"] == 8 and config.SCALE_PARAMS["embedding_dim"] == 384
    assert config.TRAIN == {"iters": 10000, "eval_iters": 200, "eval_interval": 500}


def test_gradient_bucket_plan_covers_arena():
    from drakegpt_b200.parallel import bucket_ranges
    slots, off = {}, 0
    names = ["token_embedding_table.weight", "position_embedding_table.weight"]
    names += [f"blocks.{i}.{n}" for i in range(3) for n in ("sa_head.qkv", "ffwd.net.0.weight", "ln1.weight")]
    names += ["lm_head.weight", "lm_head.bias"]
    for n in names:
        k = 100 + len(n)
        slots[n] = (off, k, (k,))
        off += (k + 63) // 64 * 64
    n_live = off
    slots["ln_f.weight"] = (off, 32, (32,))
    groups = [("lm_head.",)] + [(f"blocks.{i}.",) for i in (2, 1, 0)] + [("token_embedding_table.", "position_embedding_table.")]
    rng = bucket_ranges(slots, n_live, groups)
    assert len(rng) == 5
    covered = sorted(rng)
    assert covered[0][0] == 0 and covered[-1][1] == n_live
    assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
    with pytest.raises(ValueError):
        bucket_ranges(slots, n_live, groups[:-1])


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) prints one JSON line with the
    contract's keys, on the GPU arm's metric / unit / workload."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "train_tokens_per_sec_TransformerLM_scaled"
    assert line["unit"] == "tokens/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["config"]["workload"].startswith("TransformerLM_scaled train step") and line["config"]["seq_len"] == 256
    from oracle import stage_ref
    assert line["cpu_baseline"]["kind"] == ("reference" if stage_ref.available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["config"]["global_batch"] == 64  # timed at the GPU arm's 64x256
    assert line["e2e"] == {"value": line["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dropout_mask_restatement_matches_c_abi():
    """tests/_dropmask.py (numpy) == dgpt_dropout_keep_host (the C-ABI's host restatement of the device mask)."""
    from _dropmask import keep_mask, words
    from drakegpt_b200 import _lib
    L = _lib.lib()
    for seed, site, p in [(1234567, 3, 0.3), (2 ** 62 + 5, 0, 0.2), (99, 5, 0.25), (0, 23, 0.1)]:
        got = keep_mask((4096,), seed, site, p)
        want = torch.tensor([L.dgpt_dropout_keep_host(seed, site, i, p) for i in range(4096)], dtype=torch.float32)
        assert torch.equal(got, want)
    # far into the index space (64-bit group index), through the `start` argument
    import numpy as np
    from _dropmask import threshold
    start = (1 << 40) + 17
    w = words(7, 2, 64, start=start)
    want = [L.dgpt_dropout_keep_host(7, 2, start + i, 0.2) for i in range(64)]
    assert [(int(x) >= threshold(0.2)) for x in w] == [bool(v) for v in want]


def test_dropout_mask_pairwise_independence():
    """The 32 elements of a mask group share one 64-bit hash (even elements its low word, odd elements its high
    word) and differ only by a per-element odd multiplier and offset.  chi-square (3 dof) on the joint keep/drop
    table of EVERY pair of elements inside a group (all 496, of which the 240 same-word pairs are the critical
    ones) at p = 0.2 over 2 * 10^5 groups, the marginal keep rate of every element position, and the lag-1..4
    autocorrelation across consecutive groups."""
    import numpy as np
    from _dropmask import threshold, words
    G, p = 200000, 0.2
    keep = (words(987654321, 7, 32 * G) >= np.uint64(threshold(p))).reshape(G, 32)
    q = 1.0 - p
    rate = keep.mean(0)
    assert np.abs(rate - q).max() < 5.0 * np.sqrt(p * q / G), rate  # 5 sigma per position
    exp = G * np.array([q * q, q * p, p * q, p * p])
    worst, worst_pair = 0.0, None
    for a in range(32):
        for b in range(a + 1, 32):
            ka, kb = keep[:, a], keep[:, b]
            obs = np.array([(ka & kb).sum(), (ka & ~kb).sum(), (~ka & kb).sum(), (~ka & ~kb).sum()], dtype=np.float64)
            chi = float(((obs - exp) ** 2 / exp).sum())
            if chi > worst:
                worst, worst_pair = chi, (a, b)
    # P(chi2_3 > 27.9) = 4e-6; 496 pairs -> family-wise false-alarm rate 2e-3
    assert worst < 27.9, (worst, worst_pair)
    flat = keep.astype(np.float64) - q
    for lag in (1, 2, 3, 4):
        c = (flat[:-lag] * flat[lag:]).mean() / (p * q)
        assert abs(c) < 5.0 / np.sqrt(flat[lag:].size), (lag, c)


def test_cyclic_lr_matches_reference_trace():
    """train.cyclic_lr == torch.optim.lr_scheduler.CyclicLR(step_size_up=5, triangular) as the reference builds it
    (src/train.py:122-126); the golden trace was produced by the real scheduler."""
    from drakegpt_b200.train import cyclic_lr
    trace = load_golden("misc_vectors.pt")["cyclic_lr"]
    for step, want in enumerate(trace):
        assert abs(cyclic_lr(step, 1e-3, 5e-3) - want) < 1e-12, (step, want)


def test_oracle_matches_reference_scaled_curve_prefix():
    """The oracle port reproduces the first steps of the UNMODIFIED reference's 200-step curve at the benchmarked
    shape (tests/golden/scaled_curves.pt, dropout 0): same init, same batches, same AdamW."""
    gold = load_golden("scaled_curves.pt")
    sd = O.synthetic_state_dict("TransformerLM", seed=gold["init_seed"], **gold["cfg"])
    batches = O.structured_batches(gold["batch_seed"], 3, gold["B"], gold["T"])
    got = O.train_steps("TransformerLM", sd, batches, lr=gold["lr"], betas=gold["betas"], dropout=0.0, training=True)
    want = gold["p0.0"][0][:3]
    assert gold["p0.0"].shape == (1, 200) and gold["p0.2"].shape == (3, 200)
    assert all(abs(g - float(w)) <= 2e-5 * float(w) for g, w in zip(got, want)), (got, want.tolist())
    band = (gold["p0.2"].max(0).values - gold["p0.2"].min(0).values) / gold["p0.2"].mean(0)
    assert float(band.max()) < 0.03  # the reference's own seed-to-seed spread with dropout 0.2 (context for the GPU test)


def test_peer_optimizer_shards_tile_the_arena():
    """parallel.shard_range: 64-element aligned, contiguous, exhaustive and balanced for every world size."""
    from drakegpt_b200.parallel import shard_range
    n_live = 10_800_464 // 64 * 64 + 64 * 7
    for world in (1, 2, 3, 4, 8):
        rs = [shard_range(n_live, world, r) for r in range(world)]
        assert rs[0][0] == 0 and rs[-1][1] == n_live
        assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
        assert all(lo % 64 == 0 and hi % 64 == 0 and hi > lo for lo, hi in rs)
        sizes = [hi - lo for lo, hi in rs]
        assert max(sizes) - min(sizes) <= 64
    with pytest.raises(ValueError):
        shard_range(100, 2, 0)


def test_wgrad_split_k_follows_the_tile_policy():
    """Runner._splits mirrors launch_gemm_tc's column-tile choice for the wgrad GEMMs (engine.py / csrc/gemm_tc.cu):
    enough K splits to fill the SMs once, computed from the tile count the kernel will really use."""
    from drakegpt_b200.engine import Runner
    M, C, F, sm = 16384, 384, 1536, 148
    assert Runner._splits(F, C, M, sm) == 6            # FFN1 wgrad: 12 row tiles x 2 tiles of 192 columns
    assert Runner._splits(3 * C, C, M, sm) == 8        # QKV wgrad: 9 x 2
    assert Runner._splits(C, C, M, sm) == 16           # proj wgrad: 3 x 3 tiles of 128 (few row tiles: no 192)
    assert Runner._splits(C, F, M, sm) == 4            # FFN2 wgrad without a column sum: 3 x 12 tiles of 128
    assert Runner._splits(C, F, M, sm, colsum=True) == 8   # with the bias gradient riding on it: 3 x 6 tiles of 256
    assert Runner._splits(80, C, 64, sm) == 1          # never more splits than 512-deep K slices


def test_persistent_decoder_shape_gate_boundaries():
    """dgpt_decode_persistent_supported (host only): each limit of decode_persistent_kernel passes at its value and
    fails one step past it.  Base shape: the scaled TransformerLM (C=384, 6 heads, F=1536, V=80, 6 layers, ctx 256)."""
    from drakegpt_b200 import ops
    base = dict(B=4, nl=6, C=384, NH=6, H=64, F=1536, V=80, ctx=256, cluster=16)

    def ok(**kw):
        a = dict(base, **kw)
        return ops.decode_persistent_supported(a["B"], a["nl"], a["C"], a["NH"], a["H"], a["F"], a["V"], a["ctx"],
                                               a["cluster"])

    assert ok() and ok(cluster=0)  # 0: the default cluster of 16
    for name, at, past in [("C", 512, 520), ("F", 1536, 1544), ("V", 1536, 1537), ("nl", 8, 9), ("ctx", 256, 257),
                           ("B", 8, 9)]:
        assert ok(**{name: at}) and not ok(**{name: past}), (name, at, past)
    assert ok(C=512, NH=8, F=1536) and not ok(C=512, NH=8, F=2048)  # TransformerLM(80, 512, 256, 8, L): F = 4 C
    assert ok(C=256, NH=8, F=1024)                       # D = NH * 64 != C
    assert ok(nl=1, B=1) and not ok(nl=0) and not ok(B=0)
    assert not ok(H=32) and not ok(C=388) and not ok(F=1540)
    # the row budget: 3D (K = C) <= 12 rows x 128 warps at cluster 16, 4 rows x 64 warps of K <= 1536 at cluster 8
    assert ok(C=512, NH=8) and not ok(C=512, NH=9)
    assert ok(cluster=8, C=128, NH=2, F=512, V=80) and not ok(cluster=8)
    assert ok(cluster=4, C=64, NH=1, F=256, V=80) and not ok(cluster=4, C=128, NH=2, F=512, V=80)
    assert not ok(cluster=2) and not ok(cluster=32)
