"""Host restatement of the library's next-token rule (drakegpt_b200/csrc/sample.cuh, warp_sample_row): Philox4x32-10
as in common.cuh, then top-k, temperature, top-p and the inverse-CDF draw in fp64.  Test infrastructure only.

The device computes in fp32, so a row whose outcome hinges on a last-bit difference is reported as ambiguous rather
than compared: u within ``tol * S'`` of a boundary of the drawn token's CDF interval; a top-p cut that moves the drawn
token when the bound top_p * S moves by ``tol * S``, or two near-equal (not equal) weights at the cut; or, when the
logits themselves carry rounding noise (``logit_tol``), a k-th / (k+1)-th logit gap below it."""
import numpy as np

_M32 = 0xFFFFFFFF
SAMP = 0x53414D50  # "SAMP": third counter word of the sampling stream


def philox4x32_10(c, k):
    """Philox4x32-10 (Random123).  c: four counter words, k: two key words; each an int or a numpy uint array."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in c)
    k0, k1 = (np.asarray(x, dtype=np.uint64) for x in k)
    m32 = np.uint64(_M32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m32)
        k0 = (k0 + np.uint64(0x9E3779B9)) & m32
        k1 = (k1 + np.uint64(0xBB67AE85)) & m32
    return c0, c1, c2, c3


def uniform(b, step, seed):
    """The draw's fraction ((r.x >> 8) + 0.5) / 2^24 for rows b (int array), step and 64-bit seed."""
    b = np.asarray(b, dtype=np.uint64)
    r = philox4x32_10((b, np.full_like(b, step), np.full_like(b, SAMP), np.zeros_like(b)),
                      (seed & _M32, (seed >> 32) & _M32))
    return ((r[0] >> np.uint64(8)).astype(np.float64) + 0.5) / 2.0 ** 24


def _weights(lg, temperature, top_k):
    """Steps 1-2: (e, k-th / (k+1)-th logit gap)."""
    V = lg.shape[0]
    keep, gap = np.ones(V, dtype=bool), np.inf
    if top_k is not None and top_k < V:
        desc = np.sort(lg)[::-1]
        keep = lg >= desc[top_k - 1]
        gap = desc[top_k - 1] - desc[top_k]
    return np.where(keep, np.exp((lg - lg.max()) / temperature), 0.0), gap


def _prefix(e, top_p, slack=0.0):
    """Step 3: the (e desc, index asc) order, and the kept prefix length for the bound top_p * S + slack * S."""
    order = np.lexsort((np.arange(e.shape[0]), -e))
    eo = e[order]
    ahead = np.cumsum(eo) - eo
    return order, max(1, int((ahead < (top_p + slack) * e.sum()).sum()))


def filtered(logits, temperature=1.0, top_k=None, top_p=1.0):
    """Steps 1-3 for one row in fp64: the kept weights (0 for removed tokens)."""
    lg = np.asarray(logits, dtype=np.float64)
    e, _ = _weights(lg, temperature, top_k)
    if top_p >= 1:
        return e
    order, n = _prefix(e, top_p)
    w = np.zeros_like(e)
    w[order[:n]] = e[order[:n]]
    return w


def _inverse_cdf(w, frac, tol):
    sk = w.sum()
    u = frac * sk
    cum = np.cumsum(w)
    tok = min(int(np.searchsorted(cum, u, side="right")), len(w) - 1)
    lo = cum[tok] - w[tok]
    return tok, min(u - lo, cum[tok] - u) < tol * sk


def draw(logits, frac, temperature=1.0, top_k=None, top_p=1.0, tol=1e-5, logit_tol=0.0):
    """(token, ambiguous) for one row and the fraction of `uniform`.  With top-p, every prefix whose cut lies within
    tol * S of top_p * S is drawn from as well: the row is ambiguous unless all of them give the same token."""
    lg = np.asarray(logits, dtype=np.float64)
    e, gap = _weights(lg, temperature, top_k)
    if top_p >= 1:
        tok, amb = _inverse_cdf(e, frac, tol)
        return tok, bool(amb or gap < logit_tol)
    order, n = _prefix(e, top_p)
    _, n_lo = _prefix(e, top_p, -tol)
    _, n_hi = _prefix(e, top_p, tol)
    eo = e[order]
    amb = gap < logit_tol
    toks = set()
    for m in range(n_lo, n_hi + 1):
        if m > len(e):
            break
        w = np.zeros_like(e)
        w[order[:m]] = eo[:m]
        t, a = _inverse_cdf(w, frac, tol)
        toks.add(t)
        amb |= a
        if m < len(e) and eo[m - 1] != eo[m] and (eo[m - 1] - eo[m]) < tol * eo[m - 1]:
            amb = True  # near-equal weights at the cut may swap order in fp32
    w = np.zeros_like(e)
    w[order[:n]] = eo[:n]
    return _inverse_cdf(w, frac, tol)[0], bool(amb or len(toks) > 1)


def kept_set(logits, temperature=1.0, top_k=None, top_p=1.0):
    """Indices the rule may draw (positive kept weight)."""
    return set(np.nonzero(filtered(logits, temperature, top_k, top_p) > 0)[0].tolist())
