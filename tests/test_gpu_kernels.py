"""GPU parity of the individual C-ABI kernels against the CPU oracle's arithmetic.

Every test calls the kernels through ``drakegpt_b200.ops`` (ctypes -> C-ABI) and
compares with plain fp32 torch-CPU math on the same seeded inputs.  Exact-mode
(fp32) kernels must agree to rounding; tensor-mode (bf16 tcgen05) GEMMs are compared
on bf16-rounded operands with an fp32-accumulation tolerance.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from drakegpt_b200 import _lib, ops  # noqa: E402
from drakegpt_b200._lib import MAJOR_K, MAJOR_MN  # noqa: E402
from oracle import drake_oracle as O  # noqa: E402

DEV = "cuda"


def _keep_mask(shape, seed, site, p):
    """Host restatement of the device dropout mask (index = row-major position)."""
    n = int(torch.tensor(shape).prod())
    L = _lib.lib()
    return torch.tensor([L.dgpt_dropout_keep_host(seed, site, i, p) for i in range(n)], dtype=torch.float32).view(shape)


def test_library_loaded_and_device_ok():
    _lib.require_gpu()
    assert _lib.lib().dgpt_sm_count() >= 100


@pytest.mark.parametrize("M,N,K", [(256, 80, 32), (37, 19, 11), (64, 128, 96), (1, 5, 7)])
@pytest.mark.parametrize("amaj,bmaj", [(MAJOR_K, MAJOR_K), (MAJOR_K, MAJOR_MN), (MAJOR_MN, MAJOR_MN), (MAJOR_MN, MAJOR_K)])
def test_gemm_fp32_all_layouts(M, N, K, amaj, bmaj):
    g = torch.Generator().manual_seed(M * 1000 + N * 10 + K)
    A = torch.randn(M, K, generator=g)
    Bm = torch.randn(N, K, generator=g)
    bias = torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g)
    ref = torch.relu(A @ Bm.t() + bias) + res
    Ad = (A if amaj == MAJOR_K else A.t().contiguous()).to(DEV)
    Bd = (Bm if bmaj == MAJOR_K else Bm.t().contiguous()).to(DEV)
    out = torch.empty(M, N, device=DEV)
    ops.raw_gemm(Ad, Bd, out, a_major=amaj, b_major=bmaj, bias=bias.to(DEV), relu=True, residual=res.to(DEV))
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-5, atol=1e-5)
    # accumulate + second output
    out2 = torch.empty(M, N, device=DEV)
    ops.raw_gemm(Ad, Bd, out, a_major=amaj, b_major=bmaj, accumulate=True, out2=out2)
    torch.testing.assert_close(out.cpu(), ref + A @ Bm.t(), rtol=1e-5, atol=1e-5)


def test_gemm_fp32_dropout_and_relu_aux():
    g = torch.Generator().manual_seed(5)
    M, N, K, p, seed, site = 24, 16, 20, 0.3, 1234567, 3
    A, Bm, aux = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g), torch.randn(M, N, generator=g)
    keep = _keep_mask((M, N), seed, site, p)
    assert 0.5 < keep.mean() < 0.9
    ref = (A @ Bm.t()) * (aux > 0) * keep / (1 - p)
    out = torch.empty(M, N, device=DEV)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), out, relu_aux=aux.to(DEV), dropout=ops.Dropout(p, seed, site))
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-5, atol=1e-5)
    # device-side seed offset shifts the stream exactly like a larger host seed
    sd = torch.tensor([7], device=DEV, dtype=torch.int64)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), out, relu_aux=aux.to(DEV), dropout=ops.Dropout(p, seed - 7, site, sd))
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-5, atol=1e-5)
    # dropout_scale kernel shares the mask
    x = torch.randn(M * N, generator=g)
    y = ops.raw_dropout_scale(x.to(DEV), torch.empty(M * N, device=DEV), ops.Dropout(p, seed, site))
    torch.testing.assert_close(y.cpu(), x * keep.view(-1) / (1 - p))


TC_SHAPES = [(128, 128, 64), (256, 256, 128), (384, 1152, 384), (200, 80, 384), (130, 72, 200), (512, 384, 1536),
             (1100, 384, 128)]  # the last one: 192-column tiles (N = 384, >= 8 row tiles), ragged last row tile


@pytest.mark.parametrize("M,N,K", TC_SHAPES)
@pytest.mark.parametrize("amaj,bmaj", [(MAJOR_K, MAJOR_K), (MAJOR_K, MAJOR_MN), (MAJOR_MN, MAJOR_MN)])
def test_gemm_tcgen05_vs_fp32(M, N, K, amaj, bmaj):
    """bf16 tcgen05 GEMM == fp32 math on the same bf16-rounded operands (fp32 accumulate)."""
    g = torch.Generator().manual_seed(M + 7 * N + 13 * K)
    # MN-major operands need a 16-byte aligned row pitch: pad the leading dimension to 8 elements
    A = torch.randn(M, K, generator=g).bfloat16()
    Bm = torch.randn(N, K, generator=g).bfloat16()
    ref = A.float() @ Bm.float().t()

    def lay(X, maj):
        if maj == MAJOR_K:
            ld = (X.shape[1] + 7) // 8 * 8
            buf = torch.zeros(X.shape[0], ld, dtype=torch.bfloat16)
            buf[:, :X.shape[1]] = X
            return buf.to(DEV)[:, :X.shape[1]]
        ld = (X.shape[0] + 7) // 8 * 8
        buf = torch.zeros(X.shape[1], ld, dtype=torch.bfloat16)
        buf[:, :X.shape[0]] = X.t()
        return buf.to(DEV)[:, :X.shape[0]]

    Ad, Bd = lay(A, amaj), lay(Bm, bmaj)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.raw_gemm(Ad, Bd, out, a_major=amaj, b_major=bmaj, M=M, N=N, K=K)
    err = (out.cpu() - ref).abs().max().item()
    assert err <= 2e-3 * math.sqrt(K), (err, M, N, K, amaj, bmaj)


def test_gemm_tcgen05_epilogue_and_splitk():
    g = torch.Generator().manual_seed(21)
    M, N, K, p, seed, site = 256, 384, 512, 0.2, 99, 5
    A, Bm = torch.randn(M, K, generator=g).bfloat16(), torch.randn(N, K, generator=g).bfloat16()
    bias, res = torch.randn(N, generator=g), torch.randn(M, N, generator=g)
    acc = A.float() @ Bm.float().t()
    keep = _keep_mask((M, N), seed, site, p)
    ref = (acc + bias) * keep / (1 - p) + res
    out = torch.empty(M, N, device=DEV)
    out2 = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), out, bias=bias.to(DEV), residual=res.to(DEV), out2=out2,
                 dropout=ops.Dropout(p, seed, site))
    torch.testing.assert_close(out.cpu(), ref, rtol=1e-3, atol=5e-2)
    torch.testing.assert_close(out2.float().cpu(), ref, rtol=1e-2, atol=1e-1)
    # ReLU + bf16 output, then ReLU-mask epilogue from the saved activation
    h = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), h, bias=bias.to(DEV), relu=True)
    torch.testing.assert_close(h.float().cpu(), torch.relu(acc + bias), rtol=1e-2, atol=1e-1)
    dm = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), dm, relu_aux=h)
    torch.testing.assert_close(dm.float().cpu(), acc * (h.float().cpu() > 0), rtol=1e-2, atol=1e-1)
    # split-K wgrad-style accumulate into an fp32 gradient buffer
    Kw = 4096
    X, Y = torch.randn(Kw, 96, generator=g).bfloat16(), torch.randn(Kw, 136, generator=g).bfloat16()
    gacc = torch.ones(96, 136, device=DEV)
    ops.raw_gemm(X.to(DEV), Y.to(DEV), gacc, a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True, split_k=8)
    torch.testing.assert_close(gacc.cpu(), 1 + X.float().t() @ Y.float(), rtol=1e-3, atol=5e-2)
    # ... with the bias gradient (column sums of the stored A = dY) riding on the same GEMM
    for (Mw, Nw, sk) in [(96, 136, 8), (1536, 384, 4), (80, 384, 2)]:
        X, Y = torch.randn(Kw, Mw, generator=g).bfloat16(), torch.randn(Kw, Nw, generator=g).bfloat16()
        if Mw % 8:
            continue
        gacc = torch.ones(Mw, Nw, device=DEV)
        cs = torch.full((Mw,), 2.0, device=DEV)
        ops.raw_gemm(X.to(DEV), Y.to(DEV), gacc, a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True, split_k=sk, a_colsum=cs)
        torch.testing.assert_close(gacc.cpu(), 1 + X.float().t() @ Y.float(), rtol=1e-3, atol=5e-2)
        torch.testing.assert_close(cs.cpu(), 2 + X.float().sum(0), rtol=1e-3, atol=5e-2)


@pytest.mark.parametrize("M", [256, 200, 16384 + 96])
def test_gemm_tcgen05_residual_by_tma(M):
    """bias (+ dropout) + fp32 residual without a second output: the residual block reaches the epilogue by TMA
    (several tiles per CTA at the large M, ragged last row tile)."""
    g = torch.Generator().manual_seed(5 + M)
    N, K, p, seed, site = 384, 192, 0.2, 1234, 9
    A, Bm = torch.randn(M, K, generator=g).bfloat16(), torch.randn(N, K, generator=g).bfloat16()
    bias, res = torch.randn(N, generator=g), torch.randn(M, N, generator=g)
    acc = A.float() @ Bm.float().t()
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), out, bias=bias.to(DEV), residual=res.to(DEV))
    torch.testing.assert_close(out.cpu(), acc + bias + res, rtol=1e-3, atol=5e-2)
    if M <= 256:
        keep = _keep_mask((M, N), seed, site, p)
        out.fill_(float("nan"))
        ops.raw_gemm(A.to(DEV), Bm.to(DEV), out, bias=bias.to(DEV), residual=res.to(DEV), dropout=ops.Dropout(p, seed, site))
        torch.testing.assert_close(out.cpu(), (acc + bias) * keep / (1 - p) + res, rtol=1e-3, atol=5e-2)


@pytest.mark.parametrize("M,N", [(256, 256), (200, 1536), (384, 192)])
def test_gemm_tcgen05_relu_bit_masks(M, N):
    """Forward GEMM writes the ReLU bit mask, the dgrad GEMM applies it (== masking with the saved activation)."""
    g = torch.Generator().manual_seed(31 + N)
    K = 128
    A, Bm = torch.randn(M, K, generator=g).bfloat16(), torch.randn(N, K, generator=g).bfloat16()
    bias = torch.randn(N, generator=g)
    pre = A.float() @ Bm.float().t() + bias
    h = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    mask = torch.zeros((N // 32) * M, device=DEV, dtype=torch.int32)
    ops.raw_gemm(A.to(DEV), Bm.to(DEV), h, bias=bias.to(DEV), relu=True, relu_mask_out=mask)
    torch.testing.assert_close(h.float().cpu(), torch.relu(pre), rtol=1e-2, atol=1e-1)
    bits = (mask.cpu().view(N // 32, M, 1) >> torch.arange(32, dtype=torch.int32).view(1, 1, 32)) & 1
    got = bits.permute(1, 0, 2).reshape(M, N).bool()
    want = pre > 0
    # only values within rounding distance of zero may differ (tensor-core summation order)
    assert ((got != want) & (pre.abs() > 1e-2)).sum() == 0
    # dgrad twin: dY . W masked by the bits   (W [N, K] read MN-major as the B operand of a [M, N] x [N, K] product)
    G = torch.randn(M, K, generator=g).bfloat16()
    W2 = torch.randn(K, N, generator=g).bfloat16()  # nn.Linear(N -> K) weight: (out=K, in=N)
    d = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.raw_gemm(G.to(DEV), W2.to(DEV), d, b_major=MAJOR_MN, relu_mask_in=mask)
    ref = (G.float() @ W2.float()) * got
    torch.testing.assert_close(d.float().cpu(), ref, rtol=1e-2, atol=1e-1)
    with pytest.raises(_lib.KernelError):
        ops.raw_gemm(G.float().to(DEV), W2.float().to(DEV), torch.empty(M, N, device=DEV), b_major=MAJOR_MN, relu_mask_in=mask)


@pytest.mark.parametrize("bmaj", [MAJOR_K, MAJOR_MN])
def test_gemm_tcgen05_192_column_tiles_bf16_out(bmaj):
    """N = 384 with >= 8 row tiles runs 128 x 192 tiles; bf16 output splits the tile 128 + 64 columns between the
    two epilogue warps of a quadrant."""
    g = torch.Generator().manual_seed(192)
    M, N, K = 1300, 384, 256
    A, Bm = torch.randn(M, K, generator=g).bfloat16(), torch.randn(N, K, generator=g).bfloat16()
    Bd = (Bm if bmaj == MAJOR_K else Bm.t().contiguous()).to(DEV)
    out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16)
    ops.raw_gemm(A.to(DEV), Bd, out, b_major=bmaj, M=M, N=N, K=K)
    torch.testing.assert_close(out.float().cpu(), A.float() @ Bm.float().t(), rtol=2e-2, atol=1e-1)


def test_layernorm_fwd_bwd():
    g = torch.Generator().manual_seed(2)
    for M, C in [(64, 32), (33, 384), (5, 50)]:
        x = torch.randn(M, C, generator=g, requires_grad=True)
        w = (1 + 0.1 * torch.randn(C, generator=g)).requires_grad_()
        b = (0.1 * torch.randn(C, generator=g)).requires_grad_()
        y = torch.nn.functional.layer_norm(x, (C,), w, b, 1e-5)
        gy = torch.randn(M, C, generator=g)
        y.backward(gy)
        xd, wd, bd = (t.detach().to(DEV).requires_grad_() for t in (x, w, b))
        yd = ops.layer_norm(xd, wd, bd)
        yd.backward(gy.to(DEV))
        torch.testing.assert_close(yd.detach().cpu(), y.detach(), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(xd.grad.cpu(), x.grad, rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(wd.grad.cpu(), w.grad, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(bd.grad.cpu(), b.grad, rtol=1e-4, atol=1e-4)


def test_embedding_and_cross_entropy():
    g = torch.Generator().manual_seed(3)
    B, T, V, C = 6, 8, 80, 32
    idx = torch.randint(0, V, (B, T), generator=g)
    tgt = torch.randint(0, V, (B, T), generator=g)
    tok = torch.randn(V, C, generator=g, requires_grad=True)
    pos = torch.randn(T, C, generator=g, requires_grad=True)
    head = torch.randn(V, C, generator=g)
    x = tok[idx] + pos[torch.arange(T)]
    logits = (x @ head.t()).view(B * T, V)
    loss = torch.nn.functional.cross_entropy(logits, tgt.view(-1))
    loss.backward()
    tokd, posd = tok.detach().to(DEV).requires_grad_(), pos.detach().to(DEV).requires_grad_()
    xd = ops.embed(idx.to(DEV), tokd, posd)
    lg = ops.linear(xd, head.to(DEV)).view(B * T, V)
    ld = ops.cross_entropy(lg, tgt.view(-1).to(DEV))
    (3.0 * ld).backward()
    torch.testing.assert_close(ld.detach().cpu(), loss.detach(), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(tokd.grad.cpu(), 3 * tok.grad, rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(posd.grad.cpu(), 3 * pos.grad, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("B,T,NH,H,C", [(3, 8, 4, 8, 32), (2, 5, 1, 32, 32), (2, 64, 2, 64, 128), (1, 200, 3, 16, 48)])
def test_attention_exact_fwd_bwd(B, T, NH, H, C):
    g = torch.Generator().manual_seed(B * 100 + T)
    x = torch.randn(B, T, C, generator=g, requires_grad=True)
    w = (torch.randn(3, NH, H, C, generator=g) / math.sqrt(C)).requires_grad_()
    go = torch.randn(B, T, NH * H, generator=g)
    outs = []
    tril = torch.tril(torch.ones(T, T))
    for j in range(NH):
        sd = {"key.weight": w[1, j], "query.weight": w[0, j], "value.weight": w[2, j], "tril": tril}
        outs.append(O._one_head(sd, "", x, None, False))
    ref = torch.cat(outs, -1)
    ref.backward(go)
    xd, wd = x.detach().to(DEV).requires_grad_(), w.detach().to(DEV).requires_grad_()
    out = ops.causal_attention(xd, wd)
    out.backward(go.to(DEV))
    torch.testing.assert_close(out.detach().cpu(), ref.detach(), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(xd.grad.cpu(), x.grad, rtol=1e-3, atol=1e-5)
    torch.testing.assert_close(wd.grad.cpu(), w.grad, rtol=1e-3, atol=1e-5)


def test_attention_dropout_matches_host_mask():
    g = torch.Generator().manual_seed(8)
    B, T, NH, H, p, seed, site = 2, 6, 2, 4, 0.25, 4242, 9
    q, k, v = (torch.randn(B, T, NH * H, generator=g) for _ in range(3))
    go = torch.randn(B, T, NH * H, generator=g)
    keep = _keep_mask((B, NH, T, T), seed, site, p)
    qh, kh, vh = (t.view(B, T, NH, H).transpose(1, 2).clone().requires_grad_() for t in (q, k, v))
    s = (qh @ kh.transpose(-2, -1)) * H ** -0.5
    s = s.masked_fill(torch.tril(torch.ones(T, T)) == 0, float("-inf"))
    pd = torch.softmax(s, -1) * keep / (1 - p)
    ref = (pd @ vh).transpose(1, 2).reshape(B, T, NH * H)
    ref.backward(go)
    qd, kd, vd = q.to(DEV), k.to(DEV), v.to(DEV)
    o = torch.empty(B, T, NH * H, device=DEV)
    lse = torch.empty(B, NH, T, device=DEV)
    drop = ops.Dropout(p, seed, site)
    ops.raw_attn_fwd(qd, kd, vd, o, lse, NH, H, H ** -0.5, drop)
    torch.testing.assert_close(o.cpu(), ref.detach(), rtol=1e-4, atol=1e-5)
    dq, dk, dv = (torch.empty_like(qd) for _ in range(3))
    scratch = torch.empty((ops.attn_bwd_scratch_bytes(qd, kd, vd, o, lse, go.to(DEV), dq, dk, dv, NH, H) + 3) // 4, device=DEV)
    ops.raw_attn_bwd(qd, kd, vd, o, lse, go.to(DEV), dq, dk, dv, scratch, NH, H, H ** -0.5, drop)
    for got, want in ((dq, qh.grad), (dk, kh.grad), (dv, vh.grad)):
        torch.testing.assert_close(got.cpu(), want.transpose(1, 2).reshape(B, T, NH * H), rtol=1e-3, atol=1e-5)


@pytest.mark.parametrize("T", [128, 256])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_tcgen05_vs_exact(T, p):
    """bf16 tcgen05 attention (fwd + bwd) == exact fp32 kernel on the same bf16-rounded q,k,v,dO and mask."""
    g = torch.Generator().manual_seed(T + int(p * 10))
    B, NH, H = 2, 3, 64
    D = NH * H
    qkv = (torch.randn(B, T, 3 * D, generator=g) * 0.8).bfloat16()
    go = torch.randn(B, T, D, generator=g).bfloat16()
    drop = ops.Dropout(p, 31337, 6) if p > 0 else None
    res = {}
    for dt in (torch.float32, torch.bfloat16):
        x = qkv.to(DEV).to(dt)
        q, k, v = x[:, :, :D], x[:, :, D:2 * D], x[:, :, 2 * D:]
        o = torch.empty(B, T, D, device=DEV, dtype=dt)
        lse = torch.empty(B, NH, T, device=DEV)
        ops.raw_attn_fwd(q, k, v, o, lse, NH, H, H ** -0.5, drop)
        dx = torch.full((B, T, 3 * D), float("nan"), device=DEV, dtype=dt)
        gd = go.to(DEV).to(dt)
        scratch = torch.empty((ops.attn_bwd_scratch_bytes(q, k, v, o, lse, gd, dx[:, :, :D], dx[:, :, D:2 * D], dx[:, :, 2 * D:], NH, H) + 3) // 4, device=DEV)
        ops.raw_attn_bwd(q, k, v, o, lse, go.to(DEV).to(dt), dx[:, :, :D], dx[:, :, D:2 * D], dx[:, :, 2 * D:], scratch,
                         NH, H, H ** -0.5, drop)
        res[dt] = (o.float().cpu(), lse.cpu(), dx.float().cpu())
    (o32, l32, d32), (o16, l16, d16) = res[torch.float32], res[torch.bfloat16]
    torch.testing.assert_close(l16, l32, rtol=1e-3, atol=2e-3)
    assert (o16 - o32).abs().max() <= 3e-2, (o16 - o32).abs().max()
    assert ((o16 - o32).norm() / o32.norm()) <= 1e-2
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        a, b_ = d16[:, :, sl], d32[:, :, sl]
        assert torch.isfinite(a).all(), name
        rel = ((a - b_).norm() / b_.norm()).item()
        assert rel <= 2e-2, (name, rel)


def test_fused_adamw_matches_oracle_and_skips_frozen():
    from drakegpt_b200.optim import FlatParams, FusedAdamW
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.LayerNorm(5)).to(DEV)
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    flat = FlatParams(m, frozen=("1.",))
    flat.attach_grads()
    opt = FusedAdamW(flat, lr=3e-3)
    oracle = O.AdamW(sd, 3e-3)
    g = torch.Generator().manual_seed(1)
    for _ in range(5):
        gw, gb = torch.randn(5, 7, generator=g), torch.randn(5, generator=g)
        flat.grad("0.weight").copy_(gw)
        flat.grad("0.bias").copy_(gb)
        opt.step()
        oracle.step({"0.weight": gw, "0.bias": gb, "1.weight": None, "1.bias": None})
        assert float(flat.g.abs().sum()) == 0.0  # grads cleared by the fused kernel
    for k in sd:
        torch.testing.assert_close(m.state_dict()[k].cpu(), sd[k], rtol=1e-5, atol=1e-7)
    assert torch.equal(m.state_dict()["1.weight"].cpu(), torch.ones(5))  # frozen: no decay (SURVEY Q1/Q11)
    assert int(opt.step_dev.item()) == 5


def test_sampler_greedy_and_distribution():
    g = torch.Generator().manual_seed(4)
    Bn, V = 64, 80
    logits = torch.randn(Bn, V, generator=g) * 2
    seq = torch.zeros(Bn, 3, dtype=torch.int64, device=DEV)
    ops.raw_sample(logits.to(DEV), seq, 1, True, 0, 0)
    assert torch.equal(seq[:, 1].cpu(), logits.argmax(-1))
    assert int(seq[:, 0].abs().sum() + seq[:, 2].abs().sum()) == 0
    # one row sampled 4096 times (different batch index -> different Philox counter)
    row = torch.tensor([2.0, 1.0, 0.0, -1.0, 0.5])
    n = 4096
    big = row.repeat(n, 1).to(DEV)
    out = torch.zeros(n, 1, dtype=torch.int64, device=DEV)
    ops.raw_sample(big, out, 0, False, 777, 5)
    freq = torch.bincount(out.view(-1).cpu(), minlength=5).float() / n
    assert (freq - torch.softmax(row, -1)).abs().max() < 0.03
