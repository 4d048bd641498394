"""Time the tcgen05 GEMM at the scaled-model shapes.

Each shape is launched R times back to back inside ONE CUDA graph, every launch on its own
operand/output buffers (R sets, together larger than the 126 MB L2, so operands come from HBM as
they do inside the training step), and the graph replay is timed with CUDA events: the number is
device time per launch, free of host launch latency.  `python tools/gemm_probe.py [names...]`;
with `--single` each launch is timed alone after an L2 flush (ncu target).
"""
import sys, os, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from drakegpt_b200 import ops
from drakegpt_b200._lib import MAJOR_K, MAJOR_MN
from drakegpt_b200.engine import Runner

dev = "cuda"
shapes = {  # name: (M, N, K, a_major, b_major, out dtype, epilogue)
    "qkv_fwd": (16384, 1152, 384, MAJOR_K, MAJOR_K, torch.bfloat16, "none"),
    "proj_fwd": (16384, 384, 384, MAJOR_K, MAJOR_K, torch.float32, "bias_drop_res"),
    "ffn1_fwd": (16384, 1536, 384, MAJOR_K, MAJOR_K, torch.bfloat16, "bias_relu"),
    "ffn2_fwd": (16384, 384, 1536, MAJOR_K, MAJOR_K, torch.float32, "bias_drop_res"),
    "ffn2_dgrad": (16384, 1536, 384, MAJOR_K, MAJOR_MN, torch.bfloat16, "relu_aux"),
    "ffn1_dgrad": (16384, 384, 1536, MAJOR_K, MAJOR_MN, torch.bfloat16, "none"),
    "qkv_dgrad": (16384, 384, 1152, MAJOR_K, MAJOR_MN, torch.bfloat16, "none"),
    "proj_dgrad": (16384, 384, 384, MAJOR_K, MAJOR_MN, torch.bfloat16, "none"),
    "ffn1_wgrad": (1536, 384, 16384, MAJOR_MN, MAJOR_MN, torch.float32, "splitk"),
    "ffn2_wgrad": (384, 1536, 16384, MAJOR_MN, MAJOR_MN, torch.float32, "splitk"),
    "qkv_wgrad": (1152, 384, 16384, MAJOR_MN, MAJOR_MN, torch.float32, "splitk"),
    "proj_wgrad": (384, 384, 16384, MAJOR_MN, MAJOR_MN, torch.float32, "splitk"),
}
args = [a for a in sys.argv[1:] if not a.startswith("--")]
single = "--single" in sys.argv
which = args or list(shapes)
R = int(os.environ.get('GEMM_PROBE_R', '6'))  # operand / output sets (1: everything L2-resident)


def make(name):
    M, N, K, am, bm, odt, epi = shapes[name]
    A = torch.randn((M, K) if am == MAJOR_K else (K, M), device=dev).bfloat16()
    B = torch.randn((N, K) if bm == MAJOR_K else (K, N), device=dev).bfloat16()
    out = torch.zeros(M, N, device=dev, dtype=odt)
    kw = {}
    if epi == "bias_relu":
        kw = dict(bias=torch.zeros(N, device=dev), relu=True, relu_mask_out=torch.zeros((N // 32) * M, device=dev, dtype=torch.int32))
    elif epi == "bias_drop_res":
        kw = dict(bias=torch.zeros(N, device=dev), residual=torch.zeros(M, N, device=dev), dropout=ops.Dropout(0.2, 1, 1))
    elif epi == "relu_aux":
        kw = dict(relu_mask_in=torch.randint(-2**31, 2**31 - 1, ((N // 32) * M,), device=dev, dtype=torch.int32))
    elif epi == "splitk":
        kw = dict(accumulate=True, split_k=Runner._splits(M, N, K, ops.sm_count()))
    return lambda: ops.raw_gemm(A, B, out, a_major=am, b_major=bm, **kw)


flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
for name in which:
    M, N, K = shapes[name][:3]
    if single:
        fn = make(name)
        ts = []
        for i in range(8):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1) * 1e3)
        t = statistics.mean(ts)
    else:
        fns = [make(name) for _ in range(R)]
        for f in fns:
            f()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for rep in range(4):
                for f in fns:
                    f()
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            g.replay()
        e1.record(); e1.synchronize()
        t = e0.elapsed_time(e1) * 1e3 / (5 * 4 * R)
    print(f"{name}: {t:.1f} us  {2.0*M*N*K/t/1e6:.0f} TFLOP/s", flush=True)
