"""The fused causal attention against an fp64 restatement (tests/_attn_ref.py), at the shapes the training step runs.

The tcgen05 forward is persistent: each CTA walks a closed-form list of (batch * head, query tile) items, two in
flight, warpgroup n & 1 on item n and every mbarrier phase (n >> 1) & 1.  SHAPES reaches every regime of that
schedule (test_shapes_reach_every_forward_schedule_regime): idle CTAs, a heavy-item remainder, the leftover
round-robin of light items, 3 to 11 items on one CTA (so both warpgroups reach later items and later barrier phases),
odd item counts, and T = 128 with 3 items per CTA.  At each shape: forward and backward against fp64, the backward
issued right after the forward like in the training step.  Then dropout with a device seed offset (the engine's
per-step counter), bit-for-bit independence of the schedule, adversarial scores, and the gate that sends every
other bf16 call to the SIMT kernels, whose limits are checked too.

Bounds (each test prints its worst error as a fraction of its bound; derivations in tests/_attn_ref.py):
  * o, dq, dk, dv (bf16): |got - ref| <= half a bf16 ulp of got (the store) + the propagated error of the kernel's
    arithmetic: for O, sum_j Pd_ij |v_j| times the relative error of the kernel's probability (2^-8 for its bf16
    rounding before the P V MMA, plus the fp32 S accumulation, exp2f and the T-term sums); for dQ / dK / dV, the
    same through dS = P (dP - D) scale with the kernel's own lse and the D it computes from its own bf16 O;
  * lse (fp32): the S accumulation and exp2f errors averaged over the row's probabilities, the fp32 row sum, __logf
    and two fp32 roundings.
The SIMT kernels take the same bounds without the bf16 rounding of P / dS and with round-to-nearest accumulation."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import _attn_ref as R  # noqa: E402
from _dropmask import keep_mask  # noqa: E402
from drakegpt_b200 import _lib, ops  # noqa: E402

DEV = "cuda"
H = 64
CANARY = 7.0
SHAPES = [(1, 1, 256), (1, 6, 256), (3, 1, 128), (20, 5, 256), (25, 6, 256), (43, 7, 256), (64, 6, 256),
          (128, 6, 256), (64, 6, 128), (100, 6, 128)]
BENCH = (64, 6, 256)
MULTI = (25, 6, 256)  # 3 items on some CTAs, leftover round-robin: the adversarial inputs run here


# --------------------------------------------------------------------------- #
# the forward's schedule, restated (used to choose shapes and to name a failing item)
# --------------------------------------------------------------------------- #
def _tdiv(a, b):
    """C++ integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def _fwd_items(nheavy, nlight, G):
    """attn_fwd_tc2_kernel's item list of every CTA (csrc/attn_tc.cu, "this CTA's item list"): [[(kind, index), ...]
    per CTA] with kind "h" = query tile 1 of a T = 256 (batch, head), "l" = query tile 0; plus the heavy remainder hr
    and whether the leftover round-robin of light items runs."""
    hq, hr = nheavy // G, nheavy % G
    U = (5 * nheavy + 2 * nlight + G - 1) // G
    cap_hi, cap_lo = max(0, _tdiv(U - 5 * (hq + 1), 2)), max(0, _tdiv(U - 5 * hq, 2))
    cap_total = hr * cap_hi + (G - hr) * cap_lo
    out = []
    for c in range(G):
        nh_c = hq + (1 if c < hr else 0)
        l_start = c * cap_hi if c < hr else hr * cap_hi + (c - hr) * cap_lo
        l0, l1 = min(nlight, l_start), min(nlight, l_start + (cap_hi if c < hr else cap_lo))
        n_extra = _tdiv(nlight - cap_total - c + G - 1, G) if cap_total < nlight else 0
        lst = [("h", c + n * G) for n in range(nh_c)]
        lst += [("l", l0 + m if m < l1 - l0 else cap_total + c + (m - (l1 - l0)) * G)
                for m in range(l1 - l0 + max(0, n_extra))]
        out.append(lst)
    return out, hr, cap_total < nlight


def _schedule(B, NH, T, sm):
    bh = B * NH
    nheavy = bh if T == 256 else 0
    return _fwd_items(nheavy, bh, min(sm, nheavy + bh))


def _sm():
    sm = int(_lib.lib().dgpt_sm_count())
    assert sm > 0
    return sm


def _where(B, NH, T, b, t, h):
    """(CTA, item number, warpgroup) of the forward item that computes query row t of (b, h)."""
    items, _, _ = _schedule(B, NH, T, _sm())
    key = ("h" if T == 256 and t >= 128 else "l", b * NH + h)
    for c, lst in enumerate(items):
        if key in lst:
            n = lst.index(key)
            return dict(cta=c, item=n, warpgroup=n & 1, of=len(lst))
    return None


def test_shapes_reach_every_forward_schedule_regime():
    sm = _sm()
    reached = {}
    for B, NH, T in SHAPES:
        items, hr, leftover = _schedule(B, NH, T, sm)
        bh = B * NH
        want = sorted([("h", i) for i in range(bh if T == 256 else 0)] + [("l", i) for i in range(bh)])
        assert sorted(x for lst in items for x in lst) == want, (B, NH, T)  # every item exactly once
        n = [len(lst) for lst in items]
        for name, hit in (("idle CTAs", 0 in n), ("heavy remainder hr > 0", hr > 0), (">= 3 items", max(n) >= 3),
                          (">= 5 items", max(n) >= 5), ("odd item count > 1", any(x > 1 and x % 2 for x in n)),
                          ("leftover round-robin", leftover), ("T = 128 with >= 3 items", T == 128 and max(n) >= 3)):
            if hit:
                reached.setdefault(name, (B, NH, T))
        print(f"B={B} NH={NH} T={T}: {len(items)} CTAs, items per CTA {sorted(set(n))}, hr={hr}, leftover={leftover}")
    assert len(reached) == 7, (sm, reached)


# --------------------------------------------------------------------------- #
# helpers
# --------------------------------------------------------------------------- #
def _half_ulp(x):
    """Half a bf16 ulp of each (bf16) element of x, in fp64: the most its store can have moved it (0 stays 0)."""
    x = x.double()
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - 9))


def _qkv(B, NH, T, seed, Hh=H, amp=0.9):
    g = torch.Generator(device=DEV).manual_seed(seed)
    D = NH * Hh
    qkv = (torch.randn(B, T, 3 * D, device=DEV, generator=g) * amp).bfloat16()
    go = torch.randn(B, T, D, device=DEV, generator=g).bfloat16()
    return qkv, go


def _split(x, D):
    return x[:, :, :D], x[:, :, D:2 * D], x[:, :, 2 * D:3 * D]


def _run(q, k, v, go, NH, Hh, scale, drop=None):
    """Forward into a NaN-filled o with a padded pitch (D + 64, canary columns) and NaN-filled lse, then at once the
    backward into NaN-filled dq | dk | dv slices of one [B, T, 3D] buffer; one synchronisation at the end."""
    B, T = q.shape[:2]
    D = NH * Hh
    obuf = torch.full((B, T, D + 64), CANARY, device=DEV, dtype=torch.bfloat16)
    o = obuf[:, :, :D]
    o.fill_(float("nan"))
    lse = torch.full((B, NH, T), float("nan"), device=DEV)
    dx = torch.full((B, T, 3 * D), float("nan"), device=DEV, dtype=torch.bfloat16)
    dq, dk, dv = _split(dx, D)
    ops.raw_attn_fwd(q, k, v, o, lse, NH, Hh, scale, drop)
    nb = ops.attn_bwd_scratch_bytes(q, k, v, o, lse, go, dq, dk, dv, NH, Hh)
    scratch = torch.empty((nb + 3) // 4, device=DEV)
    ops.raw_attn_bwd(q, k, v, o, lse, go, dq, dk, dv, scratch, NH, Hh, scale, drop)
    torch.cuda.synchronize()
    assert bool((obuf[:, :, D:] == CANARY).all()), "o: pad columns overwritten"
    return dict(o=o, lse=lse, dq=dq, dk=dk, dv=dv, nb=nb)


def _ref(q, k, v, go, res, NH, Hh, scale, path, p=0.0, keep=None):
    B, T = q.shape[:2]
    heads = lambda t: t.view(B, T, NH, Hh)  # noqa: E731
    return R.reference(heads(q), heads(k), heads(v), heads(go), scale, p, keep, heads(res["o"]), res["lse"], path)


def _check(res, ref, what, shape=None):
    """Every element of o, lse, dq, dk, dv within its bound; returns the worst error / bound of each.  A NaN (an
    element the kernel did not write) fails."""
    worst = {}
    for n in ("o", "lse", "dq", "dk", "dv"):
        want, tol = ref[n], ref[n + "_tol"]
        got = res[n].double().view(want.shape)
        err = (got - want).abs() if n == "lse" else ((got - want).abs() - _half_ulp(got)).clamp_min(0)
        ratio = err / tol
        w = float(ratio.max())
        if not w <= 1.0:
            idx = tuple(int(i) for i in np.unravel_index(int(ratio.nan_to_num(float("inf")).argmax()), ratio.shape))
            b, t, h = (idx[0], idx[2], idx[1]) if n == "lse" else idx[:3]
            where = _where(*shape, b, t, h) if shape and n in ("o", "lse") else None
            raise AssertionError(f"{what} {n}: error / bound {w:.3g} at {idx} (got {float(got[idx]):.6g}, "
                                 f"want {float(want[idx]):.6g}, bound {float(tol[idx]):.3g})"
                                 + (f", forward item {where}" if where else ""))
        worst[n] = w
    print(f"{what}: worst error / bound " + " ".join(f"{n} {w:.3f}" for n, w in worst.items()))
    return worst


def _tc(B, NH, T, qkv, go, scale=H ** -0.5, drop=None, keep=None, what=""):
    D = NH * H
    q, k, v = _split(qkv, D)
    res = _run(q, k, v, go, NH, H, scale, drop)
    assert res["nb"] == 16  # the tcgen05 path: the T x T tiles never leave the chip
    ref = _ref(q, k, v, go, res, NH, H, scale, "tc", drop.p if drop else 0.0, keep)
    _check(res, ref, what or f"B={B} NH={NH} T={T}", (B, NH, T))
    return res


# --------------------------------------------------------------------------- #
# tcgen05 forward + backward at every schedule regime
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("B,NH,T", SHAPES)
def test_tcgen05_attention_vs_fp64(B, NH, T):
    """p = 0.  q | k | v are slices of one [B, T, 3D] buffer like the engine's qkv activation; o has a padded pitch
    whose pad keeps its canary; o, lse, dq, dk, dv start as NaN, so an element no item writes fails."""
    qkv, go = _qkv(B, NH, T, 100 * B + 10 * NH + T)
    _tc(B, NH, T, qkv, go)


@pytest.fixture(scope="module")
def keep_masks():
    """keep_mask restated on the host, computed once per (shape, seed) for the module, kept on the device."""
    cache = {}

    def get(shape, seed, site, p):
        key = (shape, seed, site, p)
        if key not in cache:
            cache[key] = keep_mask(shape, seed, site, p).to(DEV, torch.bool)
        return cache[key]
    return get


@pytest.mark.parametrize("B,NH,T", [BENCH, (64, 6, 128)])
def test_tcgen05_attention_dropout_device_seed_offset(B, NH, T, keep_masks):
    """p = 0.2 with the engine's form of the seed: Dropout(p, seed, site, seed_dev) with a device counter holding 7.
    Forward and backward must both use the mask of seed + 7 (element ((b NH + h) T + q) T + k), and give, bit for
    bit, what Dropout(p, seed + 7, site) without a device counter gives.  A backward that ignored the counter would
    drop other probabilities than its forward from the second training step on."""
    p, seed, site = 0.2, 20240607, 8
    qkv, go = _qkv(B, NH, T, 7 * B + T)
    ctr = torch.tensor([7], device=DEV, dtype=torch.int64)
    keep = keep_masks((B, NH, T, T), seed + 7, site, p)
    res = _tc(B, NH, T, qkv, go, drop=ops.Dropout(p, seed, site, ctr), keep=keep,
              what=f"dropout seed_dev B={B} NH={NH} T={T}")
    q, k, v = _split(qkv, NH * H)
    same = _run(q, k, v, go, NH, H, H ** -0.5, ops.Dropout(p, seed + 7, site))
    for n in ("o", "lse", "dq", "dk", "dv"):
        assert torch.equal(res[n], same[n]), n


def test_tcgen05_attention_schedule_independence():
    """Each row's arithmetic does not depend on which CTA, TMEM slot or warpgroup computes it: batches 0-1 and 62-63
    of the benchmark shape run alone as a B = 2 call (another grid, other CTAs and warpgroups) give the B = 64 call's
    o, lse, dq, dk, dv bit for bit, and so does the same B = 64 call repeated."""
    B, NH, T = BENCH
    D = NH * H
    qkv, go = _qkv(B, NH, T, 4242)
    full = _run(*_split(qkv, D), go, NH, H, H ** -0.5)
    again = _run(*_split(qkv, D), go, NH, H, H ** -0.5)
    for sl in (slice(0, 2), slice(62, 64)):
        part = _run(*_split(qkv[sl].contiguous(), D), go[sl].contiguous(), NH, H, H ** -0.5)
        for n in ("o", "lse", "dq", "dk", "dv"):
            assert torch.equal(part[n], full[n][sl]), (sl, n)
    for n in ("o", "lse", "dq", "dk", "dv"):
        assert torch.equal(again[n], full[n]), n


# --------------------------------------------------------------------------- #
# adversarial values at a shape with 3 items on some CTAs
# --------------------------------------------------------------------------- #
def _scores(qkv, NH, T, scale):
    B = qkv.shape[0]
    q, k, _ = (t.double().view(B, T, NH, H).transpose(1, 2) for t in _split(qkv, NH * H))
    return (q @ k.transpose(-1, -2)) * R.fp32_scale(scale)


@pytest.mark.parametrize("kind", ["wide", "one_key", "scale_0.3"])
def test_tcgen05_attention_adversarial(kind):
    """wide: scores spanning +-40 after scaling (the exponentials span e^80).  one_key: every query row dominated by
    one visible key chosen at random (score 20 above the rest on average), so P is nearly one-hot and O nearly one
    row of V.  scale_0.3: a scale other than H^-0.5 (not a power of two)."""
    B, NH, T = MULTI
    D = NH * H
    scale = 0.3 if kind == "scale_0.3" else H ** -0.5
    g = torch.Generator(device=DEV).manual_seed(len(kind))
    x = torch.randn(B, T, 3 * D, device=DEV, generator=g)
    q, k = x[:, :, :D].view(B, T, NH, H), x[:, :, D:2 * D].view(B, T, NH, H)
    vis = torch.ones(T, T, dtype=torch.bool, device=DEV).tril()
    if kind == "wide":
        s = _scores(x, NH, T, scale).masked_fill(~vis, 0).abs().max()
        x[:, :, :2 * D] *= float((40.0 / s) ** 0.5)
    elif kind == "one_key":
        j = (torch.rand(B, T, NH, device=DEV, generator=g) * torch.arange(1, T + 1, device=DEV).view(1, T, 1)).long()
        kj = k.gather(1, j.unsqueeze(-1).expand(B, T, NH, H))
        q.copy_(20.0 / scale * kj / kj.pow(2).sum(-1, keepdim=True) + 0.3 * q)
    qkv = x.bfloat16()
    go = torch.randn(B, T, D, device=DEV, generator=g).bfloat16()
    s = _scores(qkv, NH, T, scale).masked_fill(~vis, float("nan"))
    if kind == "wide":
        assert float(s.nan_to_num(0).max()) > 35 and float(s.nan_to_num(0).min()) < -35
    elif kind == "one_key":
        top = s.nan_to_num(float("-inf")).topk(2, -1).values
        assert float((top[..., 0] - top[..., 1])[..., 1:].median()) > 10  # the chosen key dominates
    _tc(B, NH, T, qkv, go, scale=scale, what=f"adversarial {kind}")


def test_tcgen05_attention_masks_future_keys_far_above_visible():
    """Every future key of every row scores at least 100 above every visible key of that row (score ~ 128 j plus
    noise), including the future keys inside the row's own 32-key chunk, which the forward loads and must skip
    when it takes the row maximum.  A maximum over them would underflow every visible exponential (e^-100 < 2^-126):
    a zero row sum, an infinite lse and a non-finite o."""
    B, NH, T = MULTI
    D = NH * H
    g = torch.Generator(device=DEV).manual_seed(99)
    x = torch.randn(B, T, 3 * D, device=DEV, generator=g) * 0.5
    q, k = x[:, :, :D].view(B, T, NH, H), x[:, :, D:2 * D].view(B, T, NH, H)
    q[..., 0] = 16.0
    k[..., 0] = 64.0 * torch.arange(T, device=DEV, dtype=torch.float32).view(1, T, 1)  # exact in bf16
    qkv = x.bfloat16()
    go = torch.randn(B, T, D, device=DEV, generator=g).bfloat16()
    s = _scores(qkv, NH, T, H ** -0.5)
    vis = torch.ones(T, T, dtype=torch.bool, device=DEV).tril()
    vmax = s.masked_fill(~vis, float("-inf")).amax(-1)[..., :-1]
    fmin = s.masked_fill(vis, float("inf")).amin(-1)[..., :-1]
    assert float((fmin - vmax).min()) >= 100.0
    res = _tc(B, NH, T, qkv, go, what="future keys 100 above")
    assert bool(torch.isfinite(res["lse"]).all()) and bool(torch.isfinite(res["o"].float()).all())


# --------------------------------------------------------------------------- #
# the gate: every other bf16 call runs the SIMT kernels
# --------------------------------------------------------------------------- #
GATE = ["h32", "t1", "t5", "t64", "t100", "t200", "t384", "t391", "offset", "pitch", "cache"]


@pytest.mark.parametrize("case", GATE)
def test_gate_sends_bf16_to_simt_kernels(case):
    """One violation of the tcgen05 conditions at a time, starting from the engine's aligned [B, T, 3D] layout:
    head size 32; T not in {128, 256} (T = 391 is the largest the SIMT backward's shared memory takes); a base
    one element off 16-byte alignment; a row pitch of 3D + 4 (not a multiple of 8); k / v as the first T rows of
    a longer [B, ctx, 3D] cache (batch stride != T * pitch).  Each must take the SIMT path (the exact path's scratch
    size) and match fp64 within the SIMT bounds: fp32 probabilities, round-to-nearest sums, IEEE expf / logf."""
    B, NH = 2, 6
    Hh = 32 if case == "h32" else H
    T = int(case[1:]) if case.startswith("t") else 256
    D = NH * Hh
    qkv, go = _qkv(B, NH, T, len(case) * 1000 + T, Hh)
    q, k, v = _split(qkv, D)
    if case == "offset":
        flat = torch.empty(B * T * 3 * D + 1, device=DEV, dtype=torch.bfloat16)
        shifted = flat[1:].view(B, T, 3 * D)
        shifted.copy_(qkv)
        q, k, v = _split(shifted, D)
    elif case == "pitch":
        wide = torch.zeros(B, T, 3 * D + 4, device=DEV, dtype=torch.bfloat16)
        wide[:, :, :3 * D] = qkv
        q, k, v = _split(wide, D)
    elif case == "cache":
        cache = torch.zeros(B, T + 128, 3 * D, device=DEV, dtype=torch.bfloat16)
        cache[:, :T] = qkv
        k, v = cache[:, :T, D:2 * D], cache[:, :T, 2 * D:]
    res = _run(q, k, v, go, NH, Hh, Hh ** -0.5)
    assert res["nb"] == B * NH * T * T * 8 + 16, res["nb"]
    _check(res, _ref(q, k, v, go, res, NH, Hh, Hh ** -0.5, "simt"), f"SIMT bf16 {case}")


def test_simt_backward_rejects_t_beyond_its_shared_memory():
    """The SIMT backward keeps K and V of one (batch, head) in shared memory: 584 T + 4096 bytes at H = 64, which
    caps T at 391.  At T = 392 the forward still runs (and matches fp64), the backward raises KernelError before it
    launches: dq / dk / dv keep their NaN fill and the stream stays healthy."""
    B, NH, T = 1, 1, 392
    qkv, go = _qkv(B, NH, T, 392)
    q, k, v = _split(qkv, H)
    o = torch.full((B, T, H), float("nan"), device=DEV, dtype=torch.bfloat16)
    lse = torch.full((B, NH, T), float("nan"), device=DEV)
    ops.raw_attn_fwd(q, k, v, o, lse, NH, H, H ** -0.5)
    dx = torch.full((B, T, 3 * H), float("nan"), device=DEV, dtype=torch.bfloat16)
    dq, dk, dv = _split(dx, H)
    nb = ops.attn_bwd_scratch_bytes(q, k, v, o, lse, go, dq, dk, dv, NH, H)
    assert nb == B * NH * T * T * 8 + 16
    scratch = torch.empty((nb + 3) // 4, device=DEV)
    with pytest.raises(_lib.KernelError, match="shared memory"):
        ops.raw_attn_bwd(q, k, v, o, lse, go, dq, dk, dv, scratch, NH, H, H ** -0.5)
    torch.cuda.synchronize()
    assert bool(torch.isnan(dx.float()).all())
    ref = R.reference(q.view(B, T, NH, H), k.view(B, T, NH, H), v.view(B, T, NH, H), None, H ** -0.5, path="simt")
    for n, got in (("o", o.double().view(B, T, NH, H)), ("lse", lse.double())):
        err = (got - ref[n]).abs() - (_half_ulp(got) if n == "o" else 0)
        w = float((err.clamp_min(0) / ref[n + "_tol"]).max())
        assert w <= 1.0, (n, w)
        print(f"SIMT T=392 forward {n}: worst error / bound {w:.3f}")
