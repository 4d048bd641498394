"""bench.py's headline train step with --dump-outputs: the dump is what the last timed step computed, it repeats under
the same arguments, and --steps sets how many steps are timed."""
import json
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bench(monkeypatch, capsys, out_dir, steps):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                                      "--no-cpu-baseline", "--no-kernel-table", "--dump-outputs", str(out_dir)])
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    return line, {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_bench_dump_outputs(tmp_path, monkeypatch, capsys):
    line_a, a = _bench(monkeypatch, capsys, tmp_path / "a", 2)
    line_b, b = _bench(monkeypatch, capsys, tmp_path / "b", 2)
    line_c, c = _bench(monkeypatch, capsys, tmp_path / "c", 3)
    assert (line_a["steps"], line_b["steps"], line_c["steps"]) == (2, 2, 3)
    assert sorted(a) == sorted(b) == sorted(c)
    assert len(a) == 1 + 174 and "lm_head.weight" in a and not any(k.endswith("tril") for k in a)
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert float(a["loss"]) == line_a["final_loss"]
    assert a["lm_head.weight"].shape == (80, 384) and a["blocks.5.sa_head.heads.5.key.weight"].shape == (64, 384)
    # same arguments, same inputs: the two runs differ only by the summation order of the atomically accumulated
    # gradients (an early AdamW step moves an element by about +-lr, whatever the size of its gradient, so a
    # near-zero gradient that changes sign moves it by 2 lr), far less than one more timed step moves the parameters
    assert abs(float(a["loss"]) - float(b["loss"])) <= 1e-4 * float(a["loss"])
    params = [k for k in a if k != "loss"]
    same = {k: float(np.linalg.norm(a[k] - b[k])) for k in params}
    step = {k: float(np.linalg.norm(c[k] - a[k])) for k in params}
    worst = max(params, key=lambda k: same[k] / max(step[k], 1e-30))
    assert same[worst] <= 0.5 * step[worst], (worst, same[worst], step[worst])
    assert np.sqrt(sum(v * v for v in same.values())) < 0.2 * np.sqrt(sum(v * v for v in step.values()))
    assert step["lm_head.weight"] > 0
