"""Kernel wrappers over the C-ABI plus the autograd Functions of the exact (fp32) path.

``raw_*`` functions launch one kernel on the current CUDA stream with
caller-provided tensors (no allocation unless ``out`` is omitted) and are what
the fused engine and the decoder call.  The ``torch.autograd.Function``
subclasses compose them so that the drop-in ``nn.Module`` classes in
``model_component.py`` work under ``loss.backward()``.

Nothing here computes with PyTorch ops: torch supplies device memory, streams
and the autograd tape only.
"""
import ctypes as C
import math
import numbers
import struct

import torch

from . import _lib
from ._lib import BF16, F32, MAJOR_K, MAJOR_MN, AttnArgs, GemmArgs, check

_DT = {torch.float32: F32, torch.bfloat16: BF16}


_launches = 0  # kernels enqueued through this module (bench.py reports it as gpu_launches)


def launch_count():
    return _launches


def _stream():
    global _launches
    _launches += 1
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.KernelError(
                "drakegpt_b200 ops need CUDA tensors (there is no CPU fallback); got a tensor on " + str(t.device))


def sm_count():
    """SM count of the current device (dgpt_sm_count); 148 on a B200."""
    n = int(_lib.lib().dgpt_sm_count())
    return n if n > 0 else 148


def next_seed():
    """Fresh 63-bit dropout seed from torch's CPU generator (so torch.manual_seed controls it)."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


class Dropout:
    """(p, seed, site[, seed_dev]) bundle handed to the kernels."""
    __slots__ = ("p", "seed", "site", "seed_dev")

    def __init__(self, p, seed, site=0, seed_dev=None):
        self.p, self.seed, self.site, self.seed_dev = float(p), int(seed), int(site), seed_dev


# --------------------------------------------------------------------------- #
# raw kernel launches
# --------------------------------------------------------------------------- #
def raw_gemm(A, B, out, *, a_major=MAJOR_K, b_major=MAJOR_K, M=None, N=None, K=None, bias=None, relu=False,
             relu_aux=None, dropout=None, residual=None, out2=None, accumulate=False, split_k=1,
             relu_mask_out=None, relu_mask_in=None, a_colsum=None):
    """out[M,N] = epilogue(A . B^T); see dgpt_gemm in include/drakegpt_b200.h.

    relu_mask_out / relu_mask_in: int32 tensors of (N // 32) * M words (tensor mode): the ReLU bit mask the
    forward GEMM writes and the dgrad GEMM applies.
    """
    _need_cuda(A, B, out)
    if M is None:
        M = A.shape[0] if a_major == MAJOR_K else A.shape[1]
    if K is None:
        K = A.shape[1] if a_major == MAJOR_K else A.shape[0]
    if N is None:
        N = B.shape[0] if b_major == MAJOR_K else B.shape[1]
    if A.dtype != B.dtype:
        raise _lib.KernelError(f"gemm: operand dtypes differ ({A.dtype} vs {B.dtype})")
    a = GemmArgs()
    a.A, a.B, a.D, a.D2 = _p(A), _p(B), _p(out), _p(out2)
    a.bias, a.residual, a.relu_aux = _p(bias), _p(residual), _p(relu_aux)
    a.M, a.N, a.K = M, N, K
    a.in_dtype, a.d_dtype = _DT[A.dtype], _DT[out.dtype]
    a.d2_dtype = _DT[out2.dtype] if out2 is not None else 0
    a.aux_dtype = _DT[relu_aux.dtype] if relu_aux is not None else 0
    a.a_major, a.b_major = a_major, b_major
    a.lda, a.ldb, a.ldd = A.stride(0), B.stride(0), out.stride(0)
    a.ldd2 = out2.stride(0) if out2 is not None else 0
    a.ldr = residual.stride(0) if residual is not None else 0
    a.ld_aux = relu_aux.stride(0) if relu_aux is not None else 0
    a.relu, a.accumulate, a.split_k = int(relu), int(accumulate), int(split_k)
    for mk in (relu_mask_out, relu_mask_in):
        if mk is not None and (mk.dtype != torch.int32 or mk.numel() < (N // 32) * M or not mk.is_contiguous()):
            raise _lib.KernelError("gemm: relu masks are contiguous int32 tensors of (N // 32) * M words")
    a.relu_mask_out, a.relu_mask_in = _p(relu_mask_out), _p(relu_mask_in)
    if a_colsum is not None and (a_colsum.dtype != torch.float32 or a_colsum.numel() < M):
        raise _lib.KernelError("gemm: a_colsum is an fp32 vector of M entries")
    a.a_colsum = _p(a_colsum)
    if dropout is not None and dropout.p > 0.0:
        a.dropout_p, a.seed, a.site, a.seed_dev = dropout.p, dropout.seed, dropout.site, _p(dropout.seed_dev)
    check(_lib.lib().dgpt_gemm(C.byref(a), _stream()), "dgpt_gemm")
    return out


def _attn_args(q, k, v, o, lse, NH, H, scale, dropout):
    a = AttnArgs()
    B, Tq = q.shape[0], q.shape[1]
    Tk = k.shape[1]
    a.q, a.k, a.v, a.o, a.lse = _p(q), _p(k), _p(v), _p(o), _p(lse)
    a.q_bs, a.q_rs = q.stride(0), q.stride(1)
    a.k_bs, a.k_rs = k.stride(0), k.stride(1)
    a.v_bs, a.v_rs = v.stride(0), v.stride(1)
    a.o_bs, a.o_rs = o.stride(0), o.stride(1)
    a.dtype, a.B, a.NH, a.H, a.Tq, a.Tk = _DT[q.dtype], B, NH, H, Tq, Tk
    a.scale = float(scale)
    if dropout is not None and dropout.p > 0.0:
        a.dropout_p, a.seed, a.site, a.seed_dev = dropout.p, dropout.seed, dropout.site, _p(dropout.seed_dev)
    return a


def raw_attn_fwd(q, k, v, o, lse, NH, H, scale, dropout=None):
    """q,k,v,o: [B, T, >=NH*H] views with unit inner stride; lse: [B,NH,Tq] fp32 or None."""
    _need_cuda(q, k, v, o)
    a = _attn_args(q, k, v, o, lse, NH, H, scale, dropout)
    check(_lib.lib().dgpt_attn_fwd(C.byref(a), _stream()), "dgpt_attn_fwd")
    return o


def _attn_bwd_args(q, k, v, o, lse, d_o, dq, dk, dv, scratch, NH, H, scale, dropout):
    a = _attn_args(q, k, v, o, lse, NH, H, scale, dropout)
    a.d_o, a.dq, a.dk, a.dv, a.scratch = _p(d_o), _p(dq), _p(dk), _p(dv), _p(scratch)
    a.do_bs, a.do_rs = d_o.stride(0), d_o.stride(1)
    a.dq_bs, a.dq_rs = dq.stride(0), dq.stride(1)
    a.dk_bs, a.dk_rs = dk.stride(0), dk.stride(1)
    a.dv_bs, a.dv_rs = dv.stride(0), dv.stride(1)
    return a


def attn_bwd_scratch_bytes(q, k, v, o, lse, d_o, dq, dk, dv, NH, H):
    """Scratch bytes dgpt_attn_bwd needs for exactly these operands (16 on the tcgen05 path, which keeps the
    T x T tiles on chip; B*NH*Tq*Tk*8 on the exact path).  Takes the real tensors: the kernel choice depends on
    their dtype, alignment and strides, not only on the shape."""
    a = _attn_bwd_args(q, k, v, o, lse, d_o, dq, dk, dv, None, NH, H, 1.0, None)
    return int(_lib.lib().dgpt_attn_bwd_scratch_bytes(C.byref(a)))


def raw_attn_bwd(q, k, v, o, lse, d_o, dq, dk, dv, scratch, NH, H, scale, dropout=None):
    _need_cuda(q, k, v, o, d_o, dq, dk, dv)
    a = _attn_bwd_args(q, k, v, o, lse, d_o, dq, dk, dv, scratch, NH, H, scale, dropout)
    need = int(_lib.lib().dgpt_attn_bwd_scratch_bytes(C.byref(a)))
    if scratch is None or scratch.numel() * scratch.element_size() < need:
        raise _lib.KernelError(f"attn_bwd: scratch of {need} bytes required")
    check(_lib.lib().dgpt_attn_bwd(C.byref(a), _stream()), "dgpt_attn_bwd")


def decode_attn_supported(q, k, H):
    """The bf16 KV-cache attention kernel covers head size 64 and up to 256 cached positions."""
    return q.dtype == torch.bfloat16 and H == 64 and q.shape[1] == 1 and 1 <= k.shape[1] <= 256


def raw_decode_attn(q, k, v, o, NH, H, scale):
    """One new query per (sequence, head) against the cached keys / values; see dgpt_decode_attn.
    q, o: [B, 1, >= NH*H]; k, v: [B, nk, >= NH*H] views (any batch / time strides, unit inner stride)."""
    _need_cuda(q, k, v, o)
    check(_lib.lib().dgpt_decode_attn(_p(q), _p(k), _p(v), _p(o), q.stride(0), k.stride(0), k.stride(1), v.stride(0),
                                      v.stride(1), o.stride(0), q.shape[0], NH, H, k.shape[1], float(scale), _stream()),
          "dgpt_decode_attn")
    return o


def decode_persistent_supported(B, nl, C, NH, H, F, V, ctx, cluster=0):
    """Whether the one-launch persistent decoder takes this shape (dgpt_decode_persistent_supported; cluster 0 =
    the cluster size the launch would use).  Host only: needs no device."""
    return bool(_lib.lib().dgpt_decode_persistent_supported(int(B), int(nl), int(C), int(NH), int(H), int(F), int(V),
                                                             int(ctx), int(cluster)))


def raw_embed_fwd(idx, tok, pos, x, pos_offset=0):
    _need_cuda(idx, tok, x)
    B, T = idx.shape
    V, Cdim = tok.shape
    check(_lib.lib().dgpt_embed_fwd(_p(idx), _p(tok), _p(pos), _p(x), B, T, Cdim, V, pos_offset, _stream()),
          "dgpt_embed_fwd")
    return x


def raw_embed_bwd(idx, dx, dtok, dpos, pos_offset=0):
    B, T = idx.shape
    V, Cdim = dtok.shape
    check(_lib.lib().dgpt_embed_bwd(_p(idx), _p(dx), _p(dtok), _p(dpos), B, T, Cdim, V, pos_offset, _stream()),
          "dgpt_embed_bwd")


def raw_ln_fwd(x, gamma, beta, y, mean, rstd, eps=1e-5):
    M, Cdim = x.shape
    check(_lib.lib().dgpt_ln_fwd(_p(x), _p(gamma), _p(beta), _p(y), _DT[y.dtype], _p(mean), _p(rstd), M, Cdim,
                                 float(eps), _stream()), "dgpt_ln_fwd")
    return y


def raw_embed_ln_fwd(idx, tok, pos, x, gamma, beta, y, mean, rstd, pos_offset=0, eps=1e-5):
    """x = tok[idx] + pos (written) and y = LayerNorm(x) in one pass; see dgpt_embed_ln_fwd."""
    _need_cuda(idx, tok, x, y)
    B, T = idx.shape
    V, Cdim = tok.shape
    check(_lib.lib().dgpt_embed_ln_fwd(_p(idx), _p(tok), _p(pos), _p(x), _p(gamma), _p(beta), _p(y), _DT[y.dtype],
                                       _p(mean), _p(rstd), B, T, Cdim, V, pos_offset, float(eps), _stream()),
          "dgpt_embed_ln_fwd")
    return y


def raw_ln_bwd(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, dxm=None, dropout=None, dxm_colsum=None):
    M, Cdim = x.shape
    p, seed, site, sd = 0.0, 0, 0, None
    if dropout is not None and dropout.p > 0.0:
        p, seed, site, sd = dropout.p, dropout.seed, dropout.site, _p(dropout.seed_dev)
    check(_lib.lib().dgpt_ln_bwd(_p(dy), _DT[dy.dtype], _p(x), _p(gamma), _p(mean), _p(rstd), _p(dres), _p(dx),
                                 _p(dgamma), _p(dbeta), _p(dxm), _DT[dxm.dtype] if dxm is not None else 0,
                                 _p(dxm_colsum), p, seed, sd, site, M, Cdim, _stream()), "dgpt_ln_bwd")


def raw_dropout_scale(x, out, dropout=None, relu_aux=None):
    p, seed, site, sd = 0.0, 0, 0, None
    if dropout is not None and dropout.p > 0.0:
        p, seed, site, sd = dropout.p, dropout.seed, dropout.site, _p(dropout.seed_dev)
    check(_lib.lib().dgpt_dropout_scale(_p(x), _p(relu_aux), _p(out), _DT[out.dtype], x.numel(), p, seed, sd, site,
                                        _stream()), "dgpt_dropout_scale")
    return out


def raw_cast_bf16(x, out):
    check(_lib.lib().dgpt_cast_bf16(_p(x), _p(out), x.numel(), _stream()), "dgpt_cast_bf16")
    return out


def raw_colsum(x, out, accumulate=False, M=None, N=None):
    M = x.shape[0] if M is None else M
    N = x.shape[1] if N is None else N
    check(_lib.lib().dgpt_colsum(_p(x), _DT[x.dtype], M, N, x.stride(0), _p(out), int(accumulate), _stream()),
          "dgpt_colsum")
    return out


def raw_cross_entropy(logits, targets, loss_sum, dlogits=None, dloss=None, M=None, V=None):
    M = logits.shape[0] if M is None else M
    V = logits.shape[1] if V is None else V
    check(_lib.lib().dgpt_cross_entropy(_p(logits), logits.stride(0), _p(targets), _p(loss_sum), _p(dlogits),
                                        _DT[dlogits.dtype] if dlogits is not None else 0,
                                        dlogits.stride(0) if dlogits is not None else 0, _p(dloss), M, V,
                                        _stream()), "dgpt_cross_entropy")


def lmhead_ce_supported(V, K):
    return bool(_lib.lib().dgpt_lmhead_ce_supported(int(V), int(K)))


def raw_lmhead_ce(x, w, bias, targets=None, loss_sum=None, dlogits=None, logits=None, dloss=None):
    """Fused LM head + cross-entropy (tensor mode), see dgpt_lmhead_ce: x bf16 [M,K], w bf16 [V,K]."""
    _need_cuda(x, w)
    M, K = x.shape
    V = w.shape[0]
    check(_lib.lib().dgpt_lmhead_ce(_p(x), x.stride(0), _p(w), w.stride(0), _p(bias), _p(targets), _p(loss_sum),
                                    _p(dlogits), dlogits.stride(0) if dlogits is not None else 0,
                                    _p(logits), logits.stride(0) if logits is not None else 0, _p(dloss), M, V, K,
                                    _stream()), "dgpt_lmhead_ce")


def gemm_res_ln_supported(N, K):
    return bool(_lib.lib().dgpt_gemm_res_ln_supported(int(N), int(K)))


def raw_gemm_res_ln(a, w, bias, residual, x_out, gamma, beta, y, mean, rstd, eps=1e-5, dropout=None):
    """x_out = dropout(a @ w^T + bias) + residual (fp32); y = LayerNorm(x_out) * gamma + beta (bf16); see
    dgpt_gemm_res_ln.  a bf16 [M,K], w bf16 [N,K]."""
    _need_cuda(a, w)
    M, K = a.shape
    N = w.shape[0]
    if not (a.dtype == w.dtype == y.dtype == torch.bfloat16 and residual.dtype == x_out.dtype == torch.float32):
        raise _lib.KernelError("gemm_res_ln: a / w / y must be bf16, residual / x_out fp32")
    if w.shape[1] != K or residual.shape != (M, N) or x_out.shape != (M, N) or y.shape != (M, N):
        raise _lib.KernelError(f"gemm_res_ln: shapes a {tuple(a.shape)} w {tuple(w.shape)} residual {tuple(residual.shape)} "
                          f"x_out {tuple(x_out.shape)} y {tuple(y.shape)}")
    if any(t.stride(-1) != 1 for t in (a, w, residual, x_out, y)):
        raise _lib.KernelError("gemm_res_ln: operands must be contiguous along their last dimension")
    dp, seed, site, seed_dev = 0.0, 0, 0, None
    if dropout is not None and dropout.p > 0.0:
        dp, seed, site, seed_dev = dropout.p, dropout.seed, dropout.site, dropout.seed_dev
    check(_lib.lib().dgpt_gemm_res_ln(_p(a), a.stride(0), _p(w), w.stride(0), _p(bias), _p(residual), residual.stride(0),
                                      _p(x_out), x_out.stride(0), _p(gamma), _p(beta), _p(y), y.stride(0), _p(mean),
                                      _p(rstd), M, N, K, eps, dp, seed, _p(seed_dev), site, _stream()), "dgpt_gemm_res_ln")


def raw_adamw(p, g, m, v, shadow, hyper, step, zero_grad=True, n=None):
    n = p.numel() if n is None else n
    check(_lib.lib().dgpt_adamw(_p(p), _p(g), _p(m), _p(v), _p(shadow), n, _p(hyper), _p(step), int(zero_grad),
                                _stream()), "dgpt_adamw")


def raw_counter_add(ctr, delta=1):
    check(_lib.lib().dgpt_counter_add(_p(ctr), int(delta), _stream()), "dgpt_counter_add")


def check_sampling(temperature=1.0, top_k=None, top_p=1.0):
    """Validate generate()'s sampling settings; raise ValueError before anything is launched."""
    if isinstance(temperature, bool) or not isinstance(temperature, numbers.Real) \
            or not math.isfinite(temperature) or temperature <= 0:
        raise ValueError(f"temperature must be a finite number > 0, got {temperature!r}")
    if top_k is not None and (isinstance(top_k, bool) or not isinstance(top_k, numbers.Integral) or top_k < 1):
        raise ValueError(f"top_k must be None or an int >= 1, got {top_k!r}")
    if isinstance(top_p, bool) or not isinstance(top_p, numbers.Real) or not 0 < top_p <= 1:
        raise ValueError(f"top_p must be in (0, 1], got {top_p!r}")


def sampling_settings(temperature=1.0, top_k=None, top_p=1.0):
    """Host int32[3] tensor laid out as the C-ABI's dgpt_sampling {float temperature; int32 top_k; float top_p}
    (top_k 0 = off).  Copy it into a device buffer and hand that to raw_sample / the persistent decoder.  The
    temperature is stored as float32 within [smallest normal, largest finite], so 1 / temperature stays finite."""
    check_sampling(temperature, top_k, top_p)
    t = min(max(float(temperature), 1.1754944e-38), 3.4028234e38)
    k = 0 if top_k is None else min(int(top_k), 2 ** 31 - 1)
    return torch.frombuffer(bytearray(struct.pack("<fif", t, k, float(top_p))), dtype=torch.int32).clone()


def raw_sample(logits, seq, pos, greedy, seed, step, seed_dev=None, sampling=None):
    """Next token of every row of ``logits`` into ``seq[b, pos]``.  ``sampling``: device int32[3] buffer filled from
    ``sampling_settings`` (temperature, top-k, top-p), or None for the plain softmax -> multinomial draw."""
    Bn, V = logits.shape
    if sampling is not None:
        _need_cuda(sampling)
        if sampling.dtype != torch.int32 or sampling.numel() != 3 or not sampling.is_contiguous():
            raise ValueError("raw_sample: sampling must be a contiguous int32[3] device tensor from sampling_settings")
    check(_lib.lib().dgpt_sample_ex(_p(logits), logits.stride(0), _p(seq), seq.stride(0), pos, Bn, V, int(greedy),
                                    int(seed), _p(seed_dev), int(step), _p(sampling), _stream()), "dgpt_sample_ex")


# --------------------------------------------------------------------------- #
# autograd Functions of the exact (fp32) path
# --------------------------------------------------------------------------- #
def _f32c(t):
    if t.dtype != torch.float32:
        raise _lib.KernelError(f"exact-path ops take float32 tensors, got {t.dtype}")
    return t.contiguous()


class _Embed(torch.autograd.Function):
    @staticmethod
    def forward(ctx, idx, tok, pos):
        _need_cuda(idx, tok)
        idx = idx.contiguous()
        B, T = idx.shape
        x = torch.empty((B, T, tok.shape[1]), device=tok.device, dtype=torch.float32)
        raw_embed_fwd(idx, tok.contiguous(), None if pos is None else pos.contiguous(), x)
        ctx.save_for_backward(idx)
        ctx.shapes = (tok.shape, None if pos is None else pos.shape)
        return x

    @staticmethod
    def backward(ctx, dx):
        (idx,) = ctx.saved_tensors
        tshape, pshape = ctx.shapes
        dtok = torch.zeros(tshape, device=dx.device, dtype=torch.float32)
        dpos = None if pshape is None else torch.zeros(pshape, device=dx.device, dtype=torch.float32)
        raw_embed_bwd(idx, _f32c(dx), dtok, dpos)
        return None, dtok, dpos


def embed(idx, tok, pos=None):
    """tok[idx] (+ pos[arange(T)]) -- src/model.py:595-597."""
    return _Embed.apply(idx, tok, pos)


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, residual, relu, drop):
        _need_cuda(x, w)
        shp = x.shape
        x2 = _f32c(x).view(-1, shp[-1])
        w = _f32c(w)
        M, N = x2.shape[0], w.shape[0]
        res2 = None if residual is None else _f32c(residual).view(M, N)
        y = torch.empty((M, N), device=x.device, dtype=torch.float32)
        raw_gemm(x2, w, y, bias=None if b is None else _f32c(b), relu=relu, dropout=drop, residual=res2)
        ctx.save_for_backward(x2, w, y if relu else None)
        ctx.cfg = (shp, b is not None, residual is not None, relu, drop)
        return y.view(*shp[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        x2, w, y = ctx.saved_tensors
        shp, has_b, has_res, relu, drop = ctx.cfg
        M, K = x2.shape
        N = w.shape[0]
        g = _f32c(dy).view(M, N)
        gm = g
        if relu or (drop is not None and drop.p > 0.0):
            gm = raw_dropout_scale(g, torch.empty_like(g), drop, relu_aux=y)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = raw_gemm(gm, w, torch.empty((M, K), device=g.device, dtype=torch.float32), b_major=MAJOR_MN)
            dx = dx.view(shp)
        if ctx.needs_input_grad[1]:
            dw = raw_gemm(gm, x2, torch.empty((N, K), device=g.device, dtype=torch.float32), a_major=MAJOR_MN,
                          b_major=MAJOR_MN)
        if has_b and ctx.needs_input_grad[2]:
            db = raw_colsum(gm, torch.empty((N,), device=g.device, dtype=torch.float32))
        dres = dy if has_res else None
        return dx, dw, db, dres, None, None


def linear(x, w, b=None, *, residual=None, relu=False, dropout_p=0.0, training=False):
    """residual + dropout(relu(x w^T + b)) in one GEMM epilogue (nn.Linear call sites)."""
    drop = Dropout(dropout_p, next_seed()) if (training and dropout_p > 0.0) else None
    return _Linear.apply(x, w, b, residual, relu, drop)


class _Attention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, wqkv, drop):
        _need_cuda(x, wqkv)
        B, T, Cdim = x.shape
        _, NH, H, _ = wqkv.shape
        x2 = _f32c(x).view(B * T, Cdim)
        w2 = _f32c(wqkv).view(3 * NH * H, Cdim)
        qkv = torch.empty((B * T, 3 * NH * H), device=x.device, dtype=torch.float32)
        raw_gemm(x2, w2, qkv)
        q3 = qkv.view(B, T, 3 * NH * H)
        q, k, v = q3[:, :, : NH * H], q3[:, :, NH * H: 2 * NH * H], q3[:, :, 2 * NH * H:]
        o = torch.empty((B, T, NH * H), device=x.device, dtype=torch.float32)
        lse = torch.empty((B, NH, T), device=x.device, dtype=torch.float32)
        raw_attn_fwd(q, k, v, o, lse, NH, H, H ** -0.5, drop)
        ctx.save_for_backward(x2, w2, qkv, o, lse)
        ctx.cfg = (B, T, Cdim, NH, H, drop)
        return o

    @staticmethod
    def backward(ctx, d_o):
        x2, w2, qkv, o, lse = ctx.saved_tensors
        B, T, Cdim, NH, H, drop = ctx.cfg
        d_o = _f32c(d_o)
        q3 = qkv.view(B, T, 3 * NH * H)
        q, k, v = q3[:, :, : NH * H], q3[:, :, NH * H: 2 * NH * H], q3[:, :, 2 * NH * H:]
        dqkv = torch.empty_like(qkv)
        d3 = dqkv.view(B, T, 3 * NH * H)
        dq, dk, dv = d3[:, :, : NH * H], d3[:, :, NH * H: 2 * NH * H], d3[:, :, 2 * NH * H:]
        nb = attn_bwd_scratch_bytes(q, k, v, o, lse, d_o, dq, dk, dv, NH, H)
        scratch = torch.empty((nb + 3) // 4, device=qkv.device, dtype=torch.float32)
        raw_attn_bwd(q, k, v, o, lse, d_o, dq, dk, dv, scratch, NH, H, H ** -0.5, drop)
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = raw_gemm(dqkv, w2, torch.empty_like(x2), b_major=MAJOR_MN).view(B, T, Cdim)
        if ctx.needs_input_grad[1]:
            dw = raw_gemm(dqkv, x2, torch.empty_like(w2), a_major=MAJOR_MN, b_major=MAJOR_MN).view(3, NH, H, Cdim)
        return dx, dw, None


def causal_attention(x, wqkv, *, dropout_p=0.0, training=False):
    """All heads of a causal self-attention layer: packed QKV GEMM + fused attention.

    x: (B,T,C); wqkv: (3, NH, H, C) packed as (query, key, value).  Returns
    (B, T, NH*H) with head h at columns [h*H, (h+1)*H) -- the reference's
    per-head loop + torch.cat (src/model_component.py:103,260,453).
    """
    drop = Dropout(dropout_p, next_seed()) if (training and dropout_p > 0.0) else None
    return _Attention.apply(x, wqkv, drop)


class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, eps):
        shp = x.shape
        x2 = _f32c(x).view(-1, shp[-1])
        M = x2.shape[0]
        y = torch.empty_like(x2)
        mean = torch.empty((M,), device=x.device, dtype=torch.float32)
        rstd = torch.empty((M,), device=x.device, dtype=torch.float32)
        raw_ln_fwd(x2, _f32c(w), _f32c(b), y, mean, rstd, eps)
        ctx.save_for_backward(x2, w, mean, rstd)
        ctx.shp = shp
        return y.view(shp)

    @staticmethod
    def backward(ctx, dy):
        x2, w, mean, rstd = ctx.saved_tensors
        dy2 = _f32c(dy).view_as(x2)
        dx = torch.empty_like(x2)
        dg = torch.zeros_like(w)
        db = torch.zeros_like(w)
        raw_ln_bwd(dy2, x2, _f32c(w), mean, rstd, None, dx, dg, db)
        return dx.view(ctx.shp), dg, db, None


def layer_norm(x, w, b, eps=1e-5):
    return _LayerNorm.apply(x, w, b, eps)


class _CrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, targets):
        _need_cuda(logits, targets)
        lg = _f32c(logits)
        tg = targets.contiguous()
        loss = torch.zeros((), device=lg.device, dtype=torch.float32)
        raw_cross_entropy(lg, tg, loss)
        ctx.save_for_backward(lg, tg)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        lg, tg = ctx.saved_tensors
        dl = torch.empty_like(lg)
        scratch = torch.zeros((), device=lg.device, dtype=torch.float32)
        raw_cross_entropy(lg, tg, scratch, dl, _f32c(dloss))
        return dl, None


def cross_entropy(logits, targets):
    """Mean NLL over the rows of (N, V) logits -- F.cross_entropy at src/model.py:604-607."""
    return _CrossEntropy.apply(logits, targets)
