"""The KV-cached decoders of tensor mode against an fp64 restatement (tests/_decode_ref.py), at the shapes they accept:
dgpt_decode_attn at every warps-per-(sequence, head) split with multi-chunk online softmax, the persistent decoder
through the C ABI (clusters of 4 / 8 / 16, 1-8 layers, batches 1-8, C = 512, D != C, odd V, a full 256-key context,
prompt positions after t0 > 0), its shape gate, and the engine's choice between the persistent and the per-position
path.

Tolerances (each test prints the worst error as a fraction of its bound):
  * attention output: |got - ref| <= 2^-8 |ref| + 2^-10 max|v|, the bf16 store of the output (2^-9 |ref|) plus
    fp32 / __expf accumulation;
  * KV-cache rows: |got - ref| <= 2^-8 |ref| + 2^-10 rms(row), the bf16 store of the row itself (2^-9 |ref|) plus the
    fp32 arithmetic and the rare k / v element that rounds to the other bf16 neighbour in fp32 than in fp64;
  * greedy tokens: the reference logit of the chosen token is within DELTA_P (persistent) / DELTA_G (per-position
    path, more bf16 roundings) of the reference maximum; a sampled token equals the fp64 rule's draw unless the draw
    is within EPS_LOGIT of a boundary (tests/_sampling.py)."""
import ctypes
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import _decode_ref as R  # noqa: E402
import _sampling as S  # noqa: E402
from drakegpt_b200 import _lib, ops  # noqa: E402
from drakegpt_b200 import model as M  # noqa: E402
from oracle import drake_oracle as O  # noqa: E402

DEV = "cuda"
DELTA_P = 2.0 ** -9     # persistent decoder: fp32 everywhere but the cache
# per-position path: twice its logit error bound.  An fp32 restatement of the path with its bf16 rounding points (no
# device involved) misses the fp64 logits by up to 9.1e-3 at 8 layers (C = 256), 3.9e-3 at 2 layers (C = 512): the
# rounding noise of _row_tol_g reaches the LM head.  The bound, 2^-5, is about 3 times that.
DELTA_G = 2.0 ** -4
EPS_LOGIT = 2.0 ** -12  # persistent decoder's logit error assumed by the sampling check
ROW_TOL = 2.0 ** -9     # cache rows: error beyond the bf16 store, in units of the row's rms
ATTN_TOL = 2.0 ** -12   # decode_attn: error beyond the bf16 store, in units of max |v| of the (sequence, head)
SAMPLING = (0.8, 10, 0.9)


def _half_ulp(x):
    """Half a bf16 ulp of each (bf16) element of x, in fp64: the most its store can have moved it (0 stays 0)."""
    x = x.double()
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - 9))


def _rms(ref):
    return ref.pow(2).mean(-1, keepdim=True).sqrt()


def _excess(got, ref):
    """|got - ref| beyond the rounding of got's own bf16 store, over the rms of ref's row."""
    got = got.double().cpu()
    return ((got - ref).abs() - _half_ulp(got)).clamp_min(0) / _rms(ref)


def _row_tol_g(layer):
    """ROW_TOL of the per-position path at a layer.  That path rounds to bf16 at five points per layer (LayerNorm
    outputs, q | k | v, attention output, FFN hidden).  Once its fp32 values differ from the fp64 ones by a fraction
    of an ulp, some elements round to the other bf16 neighbour, and the next layer starts from that bf16-level noise:
    the error beyond the cache's own rounding grows like sqrt(layers).  An fp32 restatement of the path with the same
    rounding points (no device involved) gives 1.0 x 2^-9 rms at layer 1 of C = 512 and 0.4, 2.2, 2.8, 2.9, 3.7, 3.7,
    4.6 x 2^-9 rms at layers 1-7 of the 8-layer C = 256 model; this bound is about 3 times that."""
    return 6.0 * math.sqrt(layer + 1) * ROW_TOL


def _check_rows(got, ref, what, tol=ROW_TOL):
    """got: bf16 cache rows, ref: their fp64 values; returns the worst excess / tol."""
    ratio = _excess(got, ref) / tol
    worst = float(ratio.max())
    assert worst <= 1.0, (what, worst, np.unravel_index(int(ratio.argmax()), ratio.shape))
    return worst


# --------------------------------------------------------------------------- #
# dgpt_decode_attn: every WPU, multi-chunk online softmax
# --------------------------------------------------------------------------- #
def _wpu(units, nk, sm):
    """dgpt_decode_attn's choice of warps per (sequence, head), restated: enough warps for one wave of 2 CTAs x 8 warps
    per SM, never more than there are 32-key chunks."""
    cap = 1 if nk <= 32 else 2 if nk <= 64 else 4 if nk <= 128 else 8
    need = 1
    while need < 8 and units * need < sm * 16:
        need *= 2
    return min(need, cap)


def _wpu_configs(sm):
    """(B, NH) giving WPU 1, 2, 4 and 8 at 256 keys."""
    out = {}
    for want, NH, units in ((1, 6, sm * 16), (2, 4, sm * 8), (4, 2, sm * 4), (8, 1, 3)):
        B = -(-units // NH)
        assert _wpu(B * NH, 256, sm) == want, (want, B, NH)
        out[want] = (B, NH)
    return out


NKS = [1, 31, 32, 33, 64, 65, 128, 129, 255, 256]


@pytest.mark.parametrize("pattern", ["random", "rising", "falling"])
@pytest.mark.parametrize("wpu", [1, 2, 4, 8])
def test_decode_attn_every_wpu_vs_fp64(wpu, pattern):
    """Scores rising along the keys make the running maximum grow at every 32-key chunk (each chunk rescales the
    partial sums by exp(old max - new max)); falling scores keep the first chunk's maximum.  Both cache layouts
    (time-major [ctx, B, 3D] and the engine's sequence-major [B, ctx, 3D]) and a padded row pitch."""
    sm = _lib.lib().dgpt_sm_count()
    assert sm > 0
    B, NH = _wpu_configs(sm)[wpu]
    H, ctx = 64, 256
    D = NH * H
    g = torch.Generator(device=DEV).manual_seed(wpu * 10 + len(pattern))
    q = torch.randn(B, NH, H, device=DEV, generator=g)
    k = torch.randn(B, ctx, NH, H, device=DEV, generator=g) * 0.7
    v = torch.randn(B, ctx, NH, H, device=DEV, generator=g) * 0.7
    if pattern != "random":
        # score(j) ~ N(0, ...) + 10 * ramp(j): a 10-unit sweep of the logits over the keys
        ramp = torch.linspace(-1.0, 1.0, ctx, device=DEV).view(1, ctx, 1, 1)
        if pattern == "falling":
            ramp = -ramp
        qn = q / q.pow(2).sum(-1, keepdim=True)  # q . qn = 1
        k = k + 10.0 * H ** 0.5 * ramp * qn.view(B, 1, NH, H)
    qb = q.bfloat16().reshape(B, D)
    kb, vb = k.bfloat16().reshape(B, ctx, D), v.bfloat16().reshape(B, ctx, D)
    pad = 3 * D + 64
    seqm = torch.zeros(B, ctx, pad, device=DEV, dtype=torch.bfloat16)  # sequence-major, padded row pitch
    seqm[:, :, D:2 * D], seqm[:, :, 2 * D:3 * D] = kb, vb
    timem = torch.zeros(ctx, B, 3 * D, device=DEV, dtype=torch.bfloat16)  # time-major
    timem[:, :, D:2 * D], timem[:, :, 2 * D:] = kb.transpose(0, 1), vb.transpose(0, 1)
    seqm[:, 0, :D] = qb  # q read from the cache row like the engine does
    worst = 0.0
    for nk in NKS:
        used = _wpu(B * NH, nk, sm)
        assert used == min(wpu, 1 if nk <= 32 else 2 if nk <= 64 else 4 if nk <= 128 else 8)
        qf = qb.double().view(B, NH, 1, H)
        kf = kb[:, :nk].double().view(B, nk, NH, H).transpose(1, 2)
        vf = vb[:, :nk].double().view(B, nk, NH, H).transpose(1, 2)
        ref = (torch.softmax(qf @ kf.transpose(-1, -2) * H ** -0.5, -1) @ vf).view(B, NH, H)
        vmax = vf.abs().amax((2, 3)).unsqueeze(-1)
        outs = []
        for name, qv, kv in (("seq-major", seqm[:, 0:1, :D], seqm[:, :nk]),
                             ("time-major", qb.view(B, 1, D), timem[:nk].transpose(0, 1))):
            out = torch.full((B, 1, D), float("nan"), device=DEV, dtype=torch.bfloat16)
            ops.raw_decode_attn(qv, kv[:, :, D:2 * D], kv[:, :, 2 * D:3 * D], out, NH, H, H ** -0.5)
            got = out.double().view(B, NH, H)
            r = float((((got - ref).abs() - _half_ulp(got)).clamp_min(0) / vmax).max()) / ATTN_TOL
            assert r <= 1.0, (name, nk, used, r)
            worst = max(worst, r)
            outs.append(out)
        assert torch.equal(outs[0], outs[1])  # the layout changes addresses only
    print(f"decode_attn WPU {wpu} {pattern} (B={B}, NH={NH}): worst excess / ATTN_TOL {worst:.3f}")


# --------------------------------------------------------------------------- #
# persistent decoder through the C ABI
# --------------------------------------------------------------------------- #
def _synthetic(C, NH, F, V, nl, ctx, seed, emb_scale=3e-3):
    """Decoder operands (D = NH * 64 may differ from C).  The embeddings are scaled so that the first LayerNorm sees a
    variance (~2e-5) comparable with its eps (1e-5): a LayerNorm that ignores eps is visibly wrong."""
    g = torch.Generator().manual_seed(seed)
    D = NH * 64

    def lin(n, k):
        return (torch.rand(n, k, generator=g) * 2 - 1) / math.sqrt(k)

    def bias(n, k):
        return (torch.rand(n, generator=g) * 2 - 1) / math.sqrt(k)

    def ln(n):
        return 1.0 + 0.05 * torch.randn(n, generator=g), 0.05 * torch.randn(n, generator=g)

    layers = []
    for _ in range(nl):
        (g1, b1_), (g2, b2_) = ln(C), ln(C)
        layers.append(dict(wqkv=lin(3 * D, C), wproj=lin(C, D), bproj=bias(C, D), w1=lin(F, C), b1=bias(F, C),
                           w2=lin(C, F), b2=bias(C, F), ln1g=g1, ln1b=b1_, ln2g=g2, ln2b=b2_))
    return dict(tok=torch.randn(V, C, generator=g) * emb_scale, pos=torch.randn(ctx, C, generator=g) * emb_scale,
                wlm=lin(V, C), blm=bias(V, C), NH=NH, layers=layers)


class _Device:
    """The persistent decoder's operands on the device, laid out like Runner._decode_persistent's."""
    ORDER = ("wqkv", "wproj", "w1", "w2", "ln1g", "ln1b", "ln2g", "ln2b", "bproj", "b1", "b2")

    def __init__(self, W, B, ctx):
        self.W, self.B, self.ctx = W, B, ctx
        bf = {"wqkv", "wproj", "w1", "w2"}
        self.layers = [{n: L[n].to(DEV, torch.bfloat16 if n in bf else torch.float32).contiguous() for n in self.ORDER}
                       for L in W["layers"]]
        self.D = W["NH"] * 64
        self.caches = [torch.empty(B, ctx, 3 * self.D, device=DEV, dtype=torch.bfloat16) for _ in W["layers"]]
        self.tok, self.pos = W["tok"].to(DEV).contiguous(), W["pos"].to(DEV).contiguous()
        self.wlm, self.blm = W["wlm"].to(DEV, torch.bfloat16).contiguous(), W["blm"].to(DEV).contiguous()
        self.seq = torch.empty(ctx + 1, B, device=DEV, dtype=torch.int64)

    def call(self, t0, t1, t_sample, greedy, seed=0, sampling=None, cluster=0):
        B = self.B
        V, C = self.W["tok"].shape
        NH, F, nl = self.W["NH"], self.W["layers"][0]["w1"].shape[0], len(self.layers)
        lib = _lib.lib()
        nfl = int(lib.dgpt_decode_persistent_scratch_floats(B, C, NH, F, V))
        scratch = torch.empty(nfl, device=DEV)
        scratch[-1] = 0.0  # barrier word
        ptrs = (ctypes.c_void_p * (12 * nl))()
        for li, L in enumerate(self.layers):
            for j, n in enumerate(self.ORDER):
                ptrs[12 * li + j] = L[n].data_ptr()
            ptrs[12 * li + 11] = self.caches[li].data_ptr()
        return lib.dgpt_decode_persistent_ex(ptrs, nl, self.tok.data_ptr(), self.pos.data_ptr(), self.wlm.data_ptr(),
                                             self.blm.data_ptr(), self.seq.data_ptr(), scratch.data_ptr(), B, C, NH,
                                             64, F, V, self.ctx, t0, t1, t_sample, int(greedy), seed, None,
                                             ops._p(sampling), cluster, ops._stream())


SENT_TOK = -7
SENT_KV = 12288.0  # exact in bf16, far outside any cache value


# name: (C, NH, F, V, layers), cluster, B, ctx, t0, t_sample, t1
PERSISTENT_CASES = {
    "C128_V97_1layer": ((128, 2, 512, 97, 1), 16, 1, 64, 0, 2, 14),
    "C256_8layers": ((256, 4, 1024, 80, 8), 16, 3, 64, 0, 1, 10),
    "C512_F1536": ((512, 8, 1536, 80, 2), 16, 4, 64, 0, 2, 12),
    "C512_F520": ((512, 8, 520, 64, 1), 16, 5, 32, 0, 3, 12),
    "D512_C256_ctx200": ((256, 8, 1024, 80, 2), 16, 7, 200, 0, 2, 12),
    "scaled_B8": ((384, 6, 1536, 80, 6), 16, 8, 256, 0, 2, 10),
    "full_context": ((128, 2, 512, 80, 2), 16, 2, 256, 0, 4, 256),
    "cluster8": ((128, 2, 512, 80, 2), 8, 3, 48, 0, 2, 12),
    "cluster4": ((64, 1, 256, 80, 2), 4, 1, 48, 0, 2, 12),
    "cluster4_B6": ((64, 1, 256, 80, 2), 4, 6, 48, 0, 2, 10),
    "prompt_after_t0": ((256, 4, 1024, 80, 2), 16, 4, 64, 6, 9, 16),
}


@pytest.mark.parametrize("case", list(PERSISTENT_CASES))
def test_persistent_decoder_vs_fp64(case):
    (C, NH, F, V, nl), cluster, B, ctx, t0, t_sample, t1 = PERSISTENT_CASES[case]
    assert ops.decode_persistent_supported(B, nl, C, NH, 64, F, V, ctx, cluster)
    W = _synthetic(C, NH, F, V, nl, ctx, seed=len(case) * 131 + C)
    dv = _Device(W, B, ctx)
    g = torch.Generator().manual_seed(C + B)
    prompt = torch.randint(0, V, (t_sample + 1, B), generator=g)
    # rows [0, t0) of the cache come from an earlier call: the reference's own (bf16) rows of the prompt
    pre_rows = R.reference(W, prompt, t0)[0] if t0 > 0 else None
    worst_rows = worst_margin = 0.0
    per_layer = {}
    n_drawn = n_ambiguous = 0
    for greedy, seed in ((True, 0), (False, 1234 + B)):
        dv.seq.fill_(SENT_TOK)
        dv.seq[:t_sample + 1] = prompt.to(DEV)
        for li, cache in enumerate(dv.caches):
            cache.fill_(SENT_KV)
            if t0 > 0:
                cache[:, :t0] = pre_rows[li].to(DEV, torch.bfloat16)
        before = [c.clone() for c in dv.caches]
        sampling = None if greedy else ops.sampling_settings(*SAMPLING).to(DEV)
        _lib.check(dv.call(t0, t1, t_sample, greedy, seed=seed, sampling=sampling, cluster=cluster), case)
        torch.cuda.synchronize()
        seq = dv.seq.cpu()
        # nothing written outside [t0, t1): the prompt, the seq rows after t1, the cache rows before t0 and from t1 on
        assert torch.equal(seq[:t_sample + 1], prompt)
        assert (seq[t1 + 1:] == SENT_TOK).all()
        assert (seq[t_sample + 1:t1 + 1] >= 0).all() and (seq[t_sample + 1:t1 + 1] < V).all()
        for li, cache in enumerate(dv.caches):
            assert torch.equal(cache[:, :t0], before[li][:, :t0]) and torch.equal(cache[:, t1:], before[li][:, t1:]), li
        rows, logits = R.reference(W, seq, t1)
        for li in range(nl):
            w = _check_rows(dv.caches[li][:, t0:t1], rows[li][:, t0:t1], (case, li))
            per_layer[li] = max(per_layer.get(li, 0.0), w)
            worst_rows = max(worst_rows, w)
        for t in range(max(t0, t_sample), t1):  # token t + 1 is drawn at position t
            lg = logits[:, t]
            tok = seq[t + 1]
            if greedy:
                short = lg.max(-1).values - lg.gather(1, tok.view(B, 1)).view(B)
                assert (short <= DELTA_P).all(), (case, t, short.tolist())
                worst_margin = max(worst_margin, float(short.max()) / DELTA_P)
            else:
                frac = S.uniform(np.arange(B), t, seed)
                for b in range(B):
                    want, amb = S.draw(lg[b].numpy(), frac[b], *SAMPLING, tol=2 * EPS_LOGIT / SAMPLING[0],
                                       logit_tol=2 * EPS_LOGIT)
                    n_drawn += 1
                    if amb:
                        n_ambiguous += 1
                        continue
                    assert int(tok[b]) == want, (case, t, b, int(tok[b]), want)
    assert n_ambiguous <= max(2, n_drawn // 5), (n_ambiguous, n_drawn)
    print(f"persistent {case}: cache rows worst excess / ROW_TOL {worst_rows:.3f}, greedy shortfall / DELTA_P "
          f"{worst_margin:.3f}, sampled {n_drawn - n_ambiguous}/{n_drawn} compared; by layer "
          f"{[round(per_layer[i], 3) for i in range(nl)]}")


# shapes around each limit: (B, nl, C, NH, F, V, ctx, cluster)
GATE_SHAPES = [(4, 6, 384, 6, 1536, 80, 256, 16), (4, 6, 512, 6, 1536, 80, 256, 16), (4, 6, 520, 6, 1536, 80, 256, 16),
               (4, 6, 384, 6, 1544, 80, 256, 16), (4, 6, 384, 6, 1536, 1536, 256, 16), (4, 6, 384, 6, 1536, 1537, 256, 16),
               (4, 8, 384, 6, 1536, 80, 256, 16), (4, 9, 384, 6, 1536, 80, 256, 16), (4, 6, 384, 6, 1536, 80, 257, 16),
               (8, 6, 384, 6, 1536, 80, 256, 16), (9, 6, 384, 6, 1536, 80, 256, 16), (1, 2, 64, 1, 256, 80, 64, 4),
               (1, 2, 128, 2, 512, 80, 64, 4), (1, 2, 128, 2, 512, 80, 64, 8), (2, 2, 512, 8, 2048, 80, 256, 16),
               (2, 2, 512, 9, 1536, 80, 256, 16), (2, 2, 384, 6, 1536, 80, 256, 2)]


def test_persistent_launch_refuses_exactly_what_the_gate_refuses():
    """dgpt_decode_persistent_ex with an empty position range checks the shape and launches nothing."""
    W = _synthetic(64, 1, 256, 80, 1, 8, seed=1)
    dv = _Device(W, 1, 8)
    lib = _lib.lib()
    dummy = torch.zeros(16, device=DEV)
    ptrs = (ctypes.c_void_p * (12 * 9))(*([dummy.data_ptr()] * (12 * 9)))
    seen = set()
    for B, nl, C, NH, F, V, ctx, cluster in GATE_SHAPES:
        ok = ops.decode_persistent_supported(B, nl, C, NH, 64, F, V, ctx, cluster)
        rc = lib.dgpt_decode_persistent_ex(ptrs, nl, dummy.data_ptr(), dummy.data_ptr(), dummy.data_ptr(),
                                           dummy.data_ptr(), dv.seq.data_ptr(), dummy.data_ptr(), B, C, NH, 64, F, V,
                                           ctx, 0, 0, 0, 1, 0, None, None, cluster, ops._stream())
        assert (rc == 0) == ok, ((B, nl, C, NH, F, V, ctx, cluster), rc, lib.dgpt_last_error())
        seen.add(ok)
    assert seen == {True, False}
    torch.cuda.synchronize()


# --------------------------------------------------------------------------- #
# the engine: which path, and both paths against the reference
# --------------------------------------------------------------------------- #
def _engine_model(vocab, C, ctx, NH, nl, seed):
    sd = O.synthetic_state_dict("TransformerLM", seed, vocab_size=vocab, embedding_dim=C, context_length=ctx,
                                num_heads=NH, num_layers=nl)
    m = M.TransformerLM(vocab, C, ctx, NH, nl, 0.0, precision="bf16")
    m.load_state_dict(sd)
    return m.to(DEV).eval(), R.weights_from_state_dict(sd)


def _engine_generate(m, W, prompt, n_new, persistent):
    """Greedy generate(); checks the tokens (margin rule) and the KV caches against the reference of the path taken.
    Returns (tokens, caches, reference rows, worst cache excess / ROW_TOL, worst shortfall / delta, last logits' error
    / delta): the per-position path leaves the logits of the last position in its workspace, the persistent decoder
    does not (None)."""
    r = m.runner()
    Bn, t0 = prompt.shape
    got = m.generate(prompt.to(DEV), n_new, greedy=True).cpu()
    assert got.shape == (Bn, t0 + n_new) and torch.equal(got[:, :t0], prompt)
    n_in = t0 + n_new - 1
    rows, logits = R.reference(W, got.t(), n_in, graph=not persistent)
    delta = DELTA_P if persistent else DELTA_G
    lg = logits[:, t0 - 1:n_in]
    short = lg.max(-1).values - lg.gather(2, got[:, t0:].unsqueeze(-1)).squeeze(-1)
    assert (short <= delta).all(), (persistent, short.max().item())
    caches, worst = [], 0.0
    for li in range(len(W["layers"])):
        D3 = 3 * W["NH"] * 64
        cache = r.buf(f"d.cache{li}", (Bn, m.context_length, D3))[:, :n_in].cpu()
        w = _check_rows(cache, rows[li], ("engine", persistent, li), ROW_TOL if persistent else _row_tol_g(li))
        print(f"  layer {li} ({'persistent' if persistent else 'per-position'}): excess / tol {w:.3f}")
        worst = max(worst, w)
        caches.append(cache)
    lerr = None
    if not persistent:
        last = r.buf("d.logits", (Bn, logits.shape[-1]), torch.float32).cpu().double()
        lerr = float((last - logits[:, n_in - 1]).abs().max()) / delta
        assert lerr <= 0.5, lerr
    return got, caches, rows, worst, float(short.max()) / delta, lerr


def test_engine_wide_model_takes_the_per_position_path():
    """TransformerLM(80, 512, 256, 8, 2): F = 4 C = 2048 is more than the persistent decoder takes, so small batches
    decode on the per-position path instead of failing."""
    m, W = _engine_model(80, 512, 256, 8, 2, seed=5)
    r = m.runner()
    for Bn in (1, 3):
        assert not r._persistent_decode_ok(Bn)
        prompt = torch.randint(0, 80, (Bn, 3), generator=torch.Generator().manual_seed(Bn))
        _, _, _, wc, ws, wl = _engine_generate(m, W, prompt, 10, persistent=False)
        print(f"engine C=512 batch {Bn}: cache worst excess / tolerance {wc:.3f}, shortfall / DELTA_G {ws:.3f}, "
              f"last logits error / DELTA_G {wl:.3f}")
    assert m.generate(prompt.to(DEV), 4).shape == (3, 7)


@pytest.mark.parametrize("shape", [(97, 128, 200, 2, 1), (80, 256, 256, 4, 8)])
def test_engine_both_paths_vs_fp64(shape, monkeypatch):
    """Shapes the persistent decoder takes, other than the scaled one: at the default batch (3) and a forced one (6)
    both paths pass the margin rule, and their KV caches agree within the two bounds."""
    vocab, C, ctx, NH, nl = shape
    m, W = _engine_model(vocab, C, ctx, NH, nl, seed=11)
    r = m.runner()
    for Bn, mode in ((3, "1"), (6, "force")):
        prompt = torch.randint(0, vocab, (Bn, 4), generator=torch.Generator().manual_seed(Bn + C))
        monkeypatch.setenv("DGPT_DECODE_PERSISTENT", mode)
        assert r._persistent_decode_ok(Bn)
        tp, cp, rp, wcp, wsp, _ = _engine_generate(m, W, prompt, 12, persistent=True)
        monkeypatch.setenv("DGPT_DECODE_PERSISTENT", "0")
        assert not r._persistent_decode_ok(Bn)
        tg, cg, rg, wcg, wsg, wlg = _engine_generate(m, W, prompt, 12, persistent=False)
        # rows of a sequence agree up to its first differing token (a near-tie may go either way)
        wpair = 0.0
        for b in range(Bn):
            diff = (tp[b] != tg[b]).nonzero()
            n = int(diff[0]) if len(diff) else tp.shape[1] - 1
            for li in range(nl):
                if n == 0:
                    continue
                a, c, ra, rc = cp[li][b, :n], cg[li][b, :n], rp[li][b, :n], rg[li][b, :n]
                # each within its bound of its own reference; the references differ by the bf16 roundings of the
                # per-position path
                slack = (a.double() - c.double()).abs() - _half_ulp(a) - _half_ulp(c) - (ra - rc).abs()
                r2 = float((slack.clamp_min(0) / _rms(rc)).max()) / (ROW_TOL + _row_tol_g(li))
                assert r2 <= 1.0, (b, li, r2)
                wpair = max(wpair, r2)
        print(f"engine {shape} batch {Bn}: persistent cache {wcp:.3f} / shortfall {wsp:.3f}; per-position cache "
              f"{wcg:.3f} / shortfall {wsg:.3f} / last logits {wlg:.3f}; the two caches {wpair:.3f} of their bound")
