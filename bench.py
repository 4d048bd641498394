#!/usr/bin/env python
"""Benchmarks of the hot path (BASELINE.json configs).

    python bench.py --gpus N --steps K --warmup W                 # config #4: TransformerLM_scaled train step (headline)
    python bench.py --impl reference --steps K --warmup W         # the UNMODIFIED reference's CPU path, same workload
    python bench.py --workload decode                             # config #5: KV-cached generation sweep, batch 1-1024
    python bench.py --workload bigram|singlehead|residual         # configs #1-#3: small-model train steps
    python bench.py --steps K --warmup W --dump-outputs DIR       # also write the headline's outputs as DIR/*.npy

One process per GPU (torchrun for N > 1, NCCL).  A "step" of the headline workload = forward + backward + gradient
reduction + AdamW on one synthetic batch of 64 x 256 tokens per GPU (weak scaling), replayed from a CUDA graph.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

S = dict(vocab_size=80, embedding_dim=384, context_length=256, num_heads=6, num_layers=6, dropout=0.2,
         batch_size=64, base_lr=3e-4)
P = dict(vocab_size=80, embedding_dim=32, context_length=8, head_size=32, num_heads=4, num_layers=3, dropout=0.1,
         batch_size=32, base_lr=1e-3)
FLOP_PER_TOKEN = 3 * (6 * (24 * 384 ** 2 + 2 * (256 + 1) * 384) + 2 * 384 * 80)  # 67 438 080 (BASELINE.md section 3)
METRIC = "train_tokens_per_sec_TransformerLM_scaled"
WORKLOAD = ("TransformerLM_scaled train step: V=80 C=384 T=256 NH=6 L=6 dropout=0.2, "
            "AdamW lr 3e-4 betas (0.9,0.95) wd 0.01; 64x256 tokens per GPU per step")
SMALL = {"bigram": "BigramLM", "singlehead": "SingleHeadAttentionLM", "residual": "ResidualBlocksLM"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"bf16_burst": p["bf16_tflops"], "bf16_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm": p["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_batches(n, B, T, V, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randint(0, V, (B, T), generator=g), torch.randint(0, V, (B, T), generator=g)) for _ in range(n)]


# --------------------------------------------------------------------------- #
# CPU arm: the reference's own implementation on the host cores
# --------------------------------------------------------------------------- #
def _reference_model(kind, cfg):
    """The unmodified reference class (oracle/_ref, staged by oracle/stage_ref.py) or None."""
    from oracle.stage_ref import load_reference
    ref = load_reference()
    if ref is None:
        return None
    C, T, V = cfg["embedding_dim"], cfg["context_length"], cfg["vocab_size"]
    if kind == "BigramLM":
        return ref.BigramLM(V)
    if kind == "SingleHeadAttentionLM":
        return ref.SingleHeadAttentionLM(V, C, T, cfg["head_size"])
    if kind == "ResidualBlocksLM":
        return ref.ResidualBlocksLM(V, C, T, cfg["num_heads"], cfg["num_layers"])
    return ref.TransformerLM(V, C, T, cfg["num_heads"], cfg["num_layers"], cfg["dropout"])


def cpu_train_tokens_per_sec(kind, cfg, B, steps, warmup, threads=None):
    """Train steps exactly as src/train.py:143-151 runs them (forward, zero_grad, backward, AdamW.step) on the host
    cores: the reference's own classes when staged (kind "reference"), else the oracle port (kind "port")."""
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    T, V = cfg["context_length"], cfg["vocab_size"]
    batches = synthetic_batches(steps + warmup, B, T, V, 42)
    torch.manual_seed(42)
    model = _reference_model(kind, cfg)
    times = []
    if model is not None:
        model.train()
        opt = torch.optim.AdamW(model.parameters(), lr=cfg["base_lr"], betas=(0.9, 0.95))
        for i, (x, y) in enumerate(batches):
            t0 = time.perf_counter()
            _, loss = model(x, y)
            opt.zero_grad()
            loss.backward()
            opt.step()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        how = "reference"
    else:
        from oracle import drake_oracle as O
        okw = {k: cfg[k] for k in ("vocab_size", "embedding_dim", "context_length", "head_size", "num_heads", "num_layers")
               if k in cfg}
        sd = O.synthetic_state_dict(kind, seed=42, **okw)
        opt = O.AdamW(sd, cfg["base_lr"])
        for i, (x, y) in enumerate(batches):
            t0 = time.perf_counter()
            _, _, grads = O.loss_and_grads(kind, sd, x, y, dropout=cfg.get("dropout", 0.0) if kind == "TransformerLM" else 0.0,
                                           training=True)
            opt.step(grads)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        how = "port"
    dt = sum(times)
    return {"value": B * T * len(times) / dt, "s_per_step": dt / len(times), "cores": torch.get_num_threads(), "kind": how,
            "steps": len(times)}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the selected workload, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "decode":
        return run_reference_decode(args)
    if args.workload in SMALL:
        kind, cfg, metric, wl = SMALL[args.workload], P, f"train_tokens_per_sec_{SMALL[args.workload]}", small_workload(args.workload)
        warmup = max(1, min(args.warmup, 5))
    else:
        kind, cfg, metric, wl = "TransformerLM", S, METRIC, WORKLOAD
        warmup = max(1, min(args.warmup, 2))  # ~4-8 s per 64x256 step on a host
    B = cfg["batch_size"]
    r = cpu_train_tokens_per_sec(kind, cfg, B, args.steps, warmup)
    sample = (f"{r['steps']} train steps (fwd+zero_grad+bwd+AdamW.step, src/train.py:143-151) of {B}x{cfg['context_length']} "
              f"tokens, fp32 torch CPU, {r['cores']} threads, "
              + ("the unmodified reference classes (oracle/_ref)" if r["kind"] == "reference" else "oracle port"))
    line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": warmup, "ms_per_step": r["s_per_step"] * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl, "global_batch": B, "seq_len": cfg["context_length"],
                       "parallelism": f"cpu{r['cores']}"},
            "cpu_baseline": {"value": r["value"], "unit": "tokens/s", "cores": r["cores"], "kind": r["kind"], "sample": sample},
            "e2e": {"value": r["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# GPU arm, headline workload (config #4)
# --------------------------------------------------------------------------- #
def roofline_dominant(dev, pk):
    """The GEMM instantiation with the largest share of the step: gemm_tc dgrad tiles at N = 384 (FFN1 / QKV / proj
    dgrad run the same instantiation; FFN1 dgrad, M=16384 N=384 K=1536, is its largest shape), launched exactly as
    the training step launches it, operands from HBM (6 rotating sets), CUDA-graph replay timed with CUDA events."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import probes
    name = "ffn1_dgrad"
    us = probes.time_launches([probes.make_gemm(name) for _ in range(probes.R)])
    tf = probes.gemm_flops(name) / us / 1e6
    traffic = None
    try:  # dram bytes of one launch from the committed `ncu --set full` capture of this kernel (profiles/)
        with open(os.path.join(ROOT, "profiles", "r2_roofline_traffic.json")) as f:
            traffic = json.load(f).get(name)
    except Exception:
        pass
    return {"bound": "tensor", "achieved": tf, "peak": pk["bf16_burst"], "unit": "TFLOP/s", "frac": tf / pk["bf16_burst"],
            "traffic": traffic, "algorithmic_bytes": probes.gemm_bytes(name), "algorithmic_flop": probes.gemm_flops(name),
            "kernel": "gemm_tc_kernel dgrad (A K-major, B MN-major, bf16 out) FFN1 dgrad 16384x384x1536, operands from HBM "
                      "(6 rotating sets); the instantiation with the largest share of the step",
            "peak_source": pk["src"] + " burst", "us_per_launch": us, "launches_timed": 5 * 4 * probes.R}


def dump_train_outputs(out_dir, model, reducer, loss, rank):
    """Write what the last step of the headline timed window hands its caller, so that two builds can be compared
    output for output: the step's loss and every parameter after its AdamW update (fp32 masters under their reference
    state_dict names, 43 MB for TransformerLM_scaled), as float32 out_dir/<name>.npy.  The fixed causal-mask buffers
    are left out."""
    if reducer is not None and getattr(reducer, "fused_optimizer", False):
        reducer.sync_master()  # each rank updated only its own shard of the fp32 masters
        torch.distributed.barrier()  # no rank starts its next step while a peer still reads its masters
    if rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array(loss, dtype=np.float32))
    for name, t in model.state_dict().items():
        if not name.endswith(".tril"):
            np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_train(args):
    from drakegpt_b200 import _lib, ops
    from drakegpt_b200 import model as M
    from drakegpt_b200.graph import GraphedTrainStep
    from drakegpt_b200.parallel import init_from_env
    import torch.distributed as dist
    rank, world, local = init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_gpu()
    pk = peaks()
    B, T, V = S["batch_size"], S["context_length"], S["vocab_size"]
    torch.manual_seed(42)
    model = M.TransformerLM(V, S["embedding_dim"], T, S["num_heads"], S["num_layers"], S["dropout"],
                            precision=args.precision).to(dev).train()
    r = model.runner()
    r.base_seed = 1000 + rank
    r.configure_optimizer(lr=S["base_lr"], betas=(0.9, 0.95))
    reducer = r.make_reducer() if world > 1 else None
    pool_host = [(x.pin_memory(), y.pin_memory()) for x, y in synthetic_batches(16, B, T, V, 42 + rank)]
    pool_dev = [(x.to(dev), y.to(dev)) for x, y in pool_host]
    n0 = ops.launch_count()
    step = GraphedTrainStep(r, B, T, reducer) if not args.no_graph else None
    launches_per_step = (ops.launch_count() - n0) // 3 if step is not None else None

    def one(i, pool):
        x, y = pool[i % len(pool)]
        if step is not None:
            return step.step(x, y)
        return r.train_step(x.to(dev, non_blocking=True), y.to(dev, non_blocking=True), reducer)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(pool, sync_each):
        for i in range(args.warmup):
            one(i, pool)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        last = 0.0
        for i in range(args.steps):
            loss = one(i, pool)
            if sync_each:
                last = loss.item()  # device -> host read of the step's loss
        e1.record()
        barrier()
        dt_dev = e0.elapsed_time(e1) * 1e-3
        dt = max(dt_dev, time.perf_counter() - t0) if sync_each else dt_dev
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), float(loss.item() if not sync_each else last)

    n1 = ops.launch_count()
    with ClockSampler(local) as cs:
        dt, loss = timed(pool_dev, sync_each=False)
    eager_launches = ops.launch_count() - n1
    clocks = cs.summary()
    if args.dump_outputs:
        dump_train_outputs(args.dump_outputs, model, reducer, loss, rank)
    dt_e2e, _ = timed(pool_host, sync_each=True)
    tokens = world * B * T * args.steps
    tps, tps_e2e = tokens / dt, tokens / dt_e2e
    if rank != 0:
        return
    roof = roofline_dominant(dev, pk)
    families = None
    if world == 1 and not args.no_kernel_table:
        import probes
        families = probes.kernel_family_table(pk)
    step_tf = tps / world * FLOP_PER_TOKEN / 1e12
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        c = cpu_train_tokens_per_sec("TransformerLM", S, B, 2, 1)
        cpu = {"value": c["value"], "unit": "tokens/s", "cores": c["cores"], "kind": c["kind"],
               "sample": f"2 train steps of {B}x256 tokens after 1 warm-up ({'unmodified reference classes, oracle/_ref' if c['kind'] == 'reference' else 'oracle port'}, "
                         f"fp32 torch CPU, {c['cores']} threads, {c['s_per_step']:.2f} s/step)"}
    gl = (launches_per_step * args.steps) if launches_per_step else eager_launches
    line = {"metric": METRIC, "value": tps, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if r.mode == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "global_batch": world * B, "seq_len": T, "parallelism": f"dp{world}",
                       "cuda_graph": step is not None,
                       "l2": "no explicit flush: each step streams > 1 GB of activations through a 126 MB L2"},
            "e2e": {"value": tps_e2e, "unit": "tokens/s", "h2d_bytes_per_step": 2 * B * T * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": gl, "launches_per_step": launches_per_step, "clocks": clocks, "roofline": roof,
            "step_tensor_frac": {"achieved_tflops_per_gpu": step_tf, "of_burst": step_tf / pk["bf16_burst"],
                                 "of_sustained": step_tf / pk["bf16_sustained"], "flop_per_token": FLOP_PER_TOKEN,
                                 "peak_source": pk["src"]},
            "kernel_families": families, "cpu_baseline": cpu, "final_loss": loss}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# configs #1-#3: small models at the PARAMS shape (32 x 8 tokens per step)
# --------------------------------------------------------------------------- #
def small_workload(w):
    return (f"{SMALL[w]} train step at the PARAMS shape (src/config.py:14-25): V=80 C=32 T=8 NH=4 L=3, AdamW lr 1e-3; "
            "32x8 tokens per step")


def run_small(args):
    """Exact fp32 CUDA-core kernels through the autograd path + the fused flat AdamW, one step per iteration
    (launch-bound at this size: 256 tokens per step; reported for completeness next to the reference's CPU path)."""
    from drakegpt_b200 import _lib, ops
    from drakegpt_b200 import model as M
    dev = torch.device("cuda", 0)
    _lib.require_gpu()
    kind = SMALL[args.workload]
    B, T, V, C = P["batch_size"], P["context_length"], P["vocab_size"], P["embedding_dim"]
    torch.manual_seed(42)
    if kind == "BigramLM":
        model = M.BigramLM(V)
    elif kind == "SingleHeadAttentionLM":
        model = M.SingleHeadAttentionLM(V, C, T, P["head_size"])
    else:
        model = M.ResidualBlocksLM(V, C, T, P["num_heads"], P["num_layers"])
    model = model.to(dev).train()
    r = model.runner()
    opt = r.configure_optimizer(lr=P["base_lr"], betas=(0.9, 0.95))
    pool_host = [(x.pin_memory(), y.pin_memory()) for x, y in synthetic_batches(16, B, T, V, 42)]
    pool_dev = [(x.to(dev), y.to(dev)) for x, y in pool_host]

    def one(x, y):
        _, loss = model(x, y)
        loss.backward()
        opt.step()
        return loss

    def timed(pool, e2e):
        for i in range(args.warmup):
            one(*[t.to(dev, non_blocking=True) for t in pool[i % 16]])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(args.steps):
            x, y = pool[i % 16]
            loss = one(x.to(dev, non_blocking=True), y.to(dev, non_blocking=True))
            if e2e:
                loss.item()
        e1.record()
        torch.cuda.synchronize()
        return max(e0.elapsed_time(e1) * 1e-3, (time.perf_counter() - t0) if e2e else 0.0)

    n0 = ops.launch_count()
    with ClockSampler(0) as cs:
        dt = timed(pool_dev, False)
    launches = ops.launch_count() - n0
    dt_e2e = timed(pool_host, True)
    tokens = B * T * args.steps
    c = cpu_train_tokens_per_sec(kind, P, B, 50, 5)
    line = {"metric": f"train_tokens_per_sec_{kind}", "value": tokens / dt, "unit": "tokens/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": small_workload(args.workload), "global_batch": B, "seq_len": T, "parallelism": "dp1",
                       "cuda_graph": False, "l2": "working set < L2 by construction (43 k parameters): launch-bound"},
            "e2e": {"value": tokens / dt_e2e, "unit": "tokens/s", "h2d_bytes_per_step": 2 * B * T * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "clocks": cs.summary(), "roofline": None,
            "cpu_baseline": {"value": c["value"], "unit": "tokens/s", "cores": c["cores"], "kind": c["kind"],
                             "sample": f"50 train steps of {B}x{T} tokens after 5 warm-up, fp32 torch CPU, {c['cores']} threads"}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# config #5: KV-cached batched generation sweep
# --------------------------------------------------------------------------- #
DECODE_WORKLOAD = ("TransformerLM_scaled KV-cached generation: prompt zeros((b,1)), 255 new tokens (inside the exact-KV "
                   "regime), softmax -> multinomial sampling on the device, batch sweep 1..1024")


def decode_byte_model(b, n_new=255):
    """BASELINE.md / SURVEY 8d: per step the bf16 weights once + KV read b*t*9216 B + KV write b*9216 B."""
    return sum(21.6e6 + b * t * 9216 + b * 9216 for t in range(n_new))


def cpu_generate_tokens_per_sec(b, n_new):
    """The reference's generate (full-window recompute per token, src/model.py:611-636) on the host cores."""
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(42)
    model = _reference_model("TransformerLM", S)
    idx = torch.zeros((b, 1), dtype=torch.long)
    if model is not None:
        model.eval()
        t0 = time.perf_counter()
        model.generate(idx, n_new)
        return b * n_new / (time.perf_counter() - t0), "reference", torch.get_num_threads()
    from oracle import drake_oracle as O
    cfg = {k: S[k] for k in ("vocab_size", "embedding_dim", "context_length", "num_heads", "num_layers")}
    sd = O.synthetic_state_dict("TransformerLM", seed=42, **cfg)
    t0 = time.perf_counter()
    O.generate("TransformerLM", sd, idx, n_new)
    return b * n_new / (time.perf_counter() - t0), "port", torch.get_num_threads()


def run_reference_decode(args):
    tps, kind, threads = cpu_generate_tokens_per_sec(16, 24)
    sample = f"generate(zeros((16,1)), 24) with the {'unmodified reference (oracle/_ref)' if kind == 'reference' else 'oracle port'}, fp32 torch CPU, {threads} threads"
    line = {"impl": "reference", "metric": "decode_tokens_per_sec_TransformerLM_scaled", "value": tps, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": 16 * 24 / tps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": DECODE_WORKLOAD, "batch": 16, "new_tokens": 24, "parallelism": f"cpu{threads}"},
            "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_decode(args):
    from drakegpt_b200 import _lib, ops
    from drakegpt_b200 import model as M
    dev = torch.device("cuda", 0)
    _lib.require_gpu()
    pk = peaks()
    torch.manual_seed(42)
    m = M.TransformerLM(S["vocab_size"], S["embedding_dim"], S["context_length"], S["num_heads"], S["num_layers"],
                        S["dropout"]).to(dev).eval()
    batches = [int(b) for b in args.decode_batches.split(",")]
    sweep = []
    n_new = 255
    launches = 0
    with ClockSampler(0) as cs:
        for b in batches:
            idx = torch.zeros((b, 1), dtype=torch.long, device=dev)
            for _ in range(max(1, min(args.warmup, 2))):
                m.generate(idx, n_new, seed=1)  # warm-up: graph capture, workspaces
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3 if b <= 64 else 1
            e0.record()
            for i in range(reps):
                out = m.generate(idx, n_new, seed=2 + i)
            e1.record()
            e1.synchronize()
            launches += ops.launch_count() - n0
            dt = e0.elapsed_time(e1) * 1e-3 / reps
            assert out.shape == (b, n_new + 1)
            # end to end: prompt from pinned host memory, generated ids read back to the host
            host_idx = torch.zeros((b, 1), dtype=torch.long).pin_memory()
            t0 = time.perf_counter()
            ids = m.generate(host_idx.to(dev, non_blocking=True), n_new, seed=9).cpu()
            dt_e2e = time.perf_counter() - t0
            gbs = decode_byte_model(b, n_new) / dt / 1e9
            sweep.append({"batch": b, "tokens_per_s": b * n_new / dt, "us_per_token_step": dt / n_new * 1e6,
                          "e2e_tokens_per_s": b * n_new / dt_e2e, "byte_model_GBps": gbs, "hbm_frac": gbs / pk["hbm"]})
            assert ids.shape == (b, n_new + 1)
    best = max(sweep, key=lambda r: r["tokens_per_s"])
    ctps, ckind, threads = (None, None, None)
    if not args.no_cpu_baseline:
        ctps, ckind, threads = cpu_generate_tokens_per_sec(16, 16)
    line = {"metric": "decode_tokens_per_sec_TransformerLM_scaled", "value": best["tokens_per_s"], "unit": "tokens/s",
            "n_gpus": 1, "steps": n_new, "warmup": args.warmup, "ms_per_step": best["us_per_token_step"] * 1e-3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": DECODE_WORKLOAD, "batch_of_value": best["batch"], "new_tokens": n_new,
                       "l2": "weights (21.6 MB bf16) are L2-resident by design; the KV cache streams from HBM at large batch"},
            "e2e": {"value": best["e2e_tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": best["batch"] * 8,
                    "d2h_bytes_per_step": best["batch"] * (n_new + 1) * 8},
            "gpu_launches": launches, "clocks": cs.summary(), "sweep": sweep,
            "roofline": {"bound": "hbm", "achieved": sweep[-1]["byte_model_GBps"], "peak": pk["hbm"], "unit": "GB/s",
                         "frac": sweep[-1]["hbm_frac"], "traffic": None,
                         "kernel": f"decode step at batch {sweep[-1]['batch']} against the weights + KV byte model",
                         "peak_source": pk["src"]},
            "cpu_baseline": None if ctps is None else {
                "value": ctps, "unit": "tokens/s", "cores": threads, "kind": ckind,
                "sample": "generate(zeros((16,1)), 16): full-window recompute per token as src/model.py:611-636"}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "decode"] + sorted(SMALL))
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16", "fp32"])
    ap.add_argument("--decode-batches", default="1,4,16,64,256,1024")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the parameters after the last step of the headline timed window as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "train"):
        ap.error("--dump-outputs writes the outputs of the GPU train step (--impl ours --workload train)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    elif args.workload == "decode":
        run_decode(args)
    else:
        run_small(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
