"""Generation sweep (BASELINE.json config #5): TransformerLM_scaled, KV-cached batched decode, 1xB200.

Prompt zeros((b,1)), 255 new tokens (stays inside the exact-KV regime, SURVEY Q12), sampling on the device.
tokens/s = b*255 / wall (CUDA events), after one warm-up call that captures the per-position graphs; with
--repeat N the median of N timed calls.  --temperature / --top-k / --top-p set the sampler (default: plain
multinomial), so the cost of the cut-offs can be measured next to the default:

    python tools/decode_bench.py 1 4 64 1024 --top-k 40 --top-p 0.9 --temperature 0.8

Also times the CPU oracle (reference semantics: full-window recompute per token) at b=1 and b=16."""
import argparse, json, os, statistics, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from drakegpt_b200 import model as M

ap = argparse.ArgumentParser()
ap.add_argument("batches", type=int, nargs="*", default=[1, 4, 16, 64, 256, 1024])
ap.add_argument("--temperature", type=float, default=1.0)
ap.add_argument("--top-k", type=int, default=None)
ap.add_argument("--top-p", type=float, default=1.0)
ap.add_argument("--repeat", type=int, default=1)
args = ap.parse_args()
samp = dict(temperature=args.temperature, top_k=args.top_k, top_p=args.top_p)
dev = "cuda"
torch.manual_seed(42)
m = M.TransformerLM(80, 384, 256, 6, 6, 0.2).to(dev).eval()
rows = []
for b in args.batches:
    idx = torch.zeros((b, 1), dtype=torch.long, device=dev)
    m.generate(idx, 255, seed=1, **samp)  # warm-up / graph capture
    torch.cuda.synchronize()
    times = []
    for i in range(args.repeat):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = m.generate(idx, 255, seed=2 + i, **samp)
        e1.record(); e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
        assert out.shape == (b, 256)
    dt = statistics.median(times)
    # byte model (BASELINE.md): weights once per step (bf16) + KV read b*t*9216 + KV write b*9216
    bytes_total = sum(21.6e6 + b * t * 9216 + b * 9216 for t in range(255))
    rows.append({"batch": b, **samp, "tokens_per_s": b * 255 / dt, "ms_per_token_step": dt / 255 * 1e3,
                 "model_GBps": bytes_total / dt / 1e9, "repeat": args.repeat})
    print(json.dumps(rows[-1]), flush=True)
if "--cpu" in os.environ.get("DECODE_BENCH", ""):
    from oracle import drake_oracle as O
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    for b, n in ((1, 32), (16, 16)):
        t0 = time.perf_counter()
        O.generate("TransformerLM", sd, torch.zeros((b, 1), dtype=torch.long), n)
        dt = time.perf_counter() - t0
        print(json.dumps({"cpu_oracle_batch": b, "tokens_per_s": b * n / dt, "threads": torch.get_num_threads()}), flush=True)
