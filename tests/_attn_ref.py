"""fp64 restatement of the fused causal attention (csrc/attn_tc.cu, csrc/attn_simt.cu) and the most each kernel may
differ from it.  Test infrastructure only: plain torch ops in fp64, on whatever device the inputs live on, no project
kernel.

Notation, per (batch, head) and query row i, key j <= i (masked keys contribute nothing):
  S_ij = s q_i.k_j, s the fp32 scale the kernels receive;  P = softmax_j(S);  lse_i = logsumexp_j(S_ij);
  M = keep / (1 - p) (1 without dropout);  Pd = P o M;  O = Pd V;  dP = dO V^T;  D_i = sum_j Pd_ij dP_ij = dO_i.O_i;
  dS = P o (dP o M - D) s;  dQ = dS K;  dK = dS^T Q;  dV = Pd^T dO.
The inputs are the bf16 values the kernels read, so every product of two inputs is exact in fp32 and the errors are
those of the kernels' own arithmetic:
  * an n-term fp32 sum is off by at most n u sum|terms|, with u = 2^-24 for round-to-nearest (the SIMT kernels' fmaf
    chains) and u = 2^-23 for the tensor-core accumulators, whose rounding is not specified as round-to-nearest;
  * S and dP are H-term sums:  |dS_raw_ij| <= H u A_ij with A = s |Q| |K|^T, and H u B_ij with B = |dO| |V|^T;
  * exp2f / expf and the rounding of their argument: the tcgen05 kernels build with --use_fast_math, where exp2f is
    ex2.approx.ftz.f32 (2 ulp) and logf is __logf (2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere).  One exponential
    of the row is then off by a relative delta_ij = H u A_ij + 2^-21 (|S_ij| + |m_i|) + 2^-21: the S error, the
    fp32 roundings of S * scale * log2(e) and of the subtraction of the row maximum m (up to 4 of 2^-24 each, times
    ln 2 for the natural-log units), and 4 ulp for the exponential itself;
  * normalising by the kernel's own row sum cancels the part of the errors common to the row: the kernel's
    probability is P_ij exp(+-(delta_ij + dbar_i)) with dbar_i = log(1 + sum_j P_ij expm1(delta_ij)) (Jensen), so
    |P~ - P| <= P eps with eps = expm1(delta + dbar);
  * tcgen05 rounds P (forward, before P V) and Pd and dS (backward, before the second-stage MMAs) to bf16.  bf16
    carries 8 significant bits, so rounding to nearest moves a value by up to half an ulp = 2^-8 of it (just above
    a power of two; 2^-9 just below one): r = 2^-8.  The SIMT kernels keep them in fp32 (r = 0);
  * values below 2^-126 flush to zero under --use_fast_math.  With operands below 2^14 and at most 2^9 keys, what
    they drop is below 2^-126 2^9 2^28 = 2^-89 per output element: FLOOR covers it.
Each bound below is the propagation of these through the kernel's formula, to all orders where the factors multiply
((1 + a)(1 + b) - 1 rather than a + b).  The bf16 store of each output is not in these bounds: the tests add half an
ulp of the stored value (tests/test_gpu_attention.py).

  forward   |O~ - O| <= sum_j Pd_ij |v_j| ((1 + sig)(1 + T u)(1 + eps_ij)(1 + r) - 1):  the kernel's probability, its
            bf16 rounding, the T-term P V sum and sig, the row sum (T terms) with 1 / sum, 1 / (1 - p) and the scaling;
            |lse~ - lse| <= dbar_i + T 2^-24 + 2^-21 (1 + |lse - m|) + 2^-22 (|m| + |lse|):  the exponentials (as
            above), the row sum, __logf of it and the fp32 roundings of m * scale and of the final add.
  backward  the kernel recomputes P from its own lse~, so delta^b_ij = H u A_ij + 2^-21 (|S_ij| + |lse_i|) + 2^-21 +
            |lse~_i - lse_i| and eps^b = expm1(delta^b) (no renormalisation); dP o M is off by
            e_ij = (H u B_ij + 2^-23 |dP_ij|) M_ij (the H-term sum, 1 / (1 - p) and the product);
            D is off by dD_i:  tcgen05 computes it from the kernel's bf16 O~ and dO:
            |dO_i.(O~_i - O_i)| + H 2^-24 sum_d |dO_id O~_id|;  SIMT sums P~ (dP o M)~ over T keys in fp32;
            dS is then off by E = s P (eps^b |dP o M - D| + (1 + eps^b)(e + dD))(1 + 2^-22) + 2^-22 |dS| (three fp32
            operations), and after the bf16 rounding and the T-term second-stage sums
            |dQ~ - dQ| <= G |K|, |dK~ - dK| <= G^T |Q|, G = ((1 + r)(1 + T u) - 1) |dS| + (1 + r)(1 + T u) E;
            |dV~ - dV| <= (Pd ((1 + eps^b)(1 + 2^-23)(1 + r)(1 + T u) - 1))^T |dO|.
"""
import torch

F64 = torch.float64
U24 = 2.0 ** -24
EXP = 2.0 ** -21
FLOOR = 2.0 ** -80
PATHS = {"tc": (2.0 ** -23, 2.0 ** -8),  # (u of the accumulators, rounding of P / Pd / dS before an MMA)
         "simt": (2.0 ** -24, 0.0)}


def fp32_scale(scale):
    """The scale as the kernels see it (the C ABI takes a float)."""
    return float(torch.tensor(scale, dtype=torch.float32))


def reference(q, k, v, d_o, scale, p=0.0, keep=None, o_got=None, lse_got=None, path="tc", chunk=8):
    """q, k, v, d_o, o_got: [B, T, NH, H] (the kernels' operands, any float dtype); keep: [B, NH, T, T] (1 = kept) or
    None; lse_got: [B, NH, T].  o_got / lse_got are the kernel's forward outputs, which its backward reads: they are
    needed for the backward bounds only.  Returns a dict of fp64 tensors on q's device: o, o_tol [B, T, NH, H];
    lse, lse_tol [B, NH, T]; with d_o also dq, dk, dv and their *_tol [B, T, NH, H].  Chunked over the batch."""
    B, T, NH, H = q.shape
    u, r = PATHS[path]
    s = fp32_scale(scale)
    inv_keep = 1.0 / (1.0 - p)
    vis = torch.ones(T, T, dtype=torch.bool, device=q.device).tril()
    cS, cT, c24 = H * u, T * u, T * U24
    sig = c24 + 2.0 ** -20
    out = {}

    def put(name, t, lay=True):
        out.setdefault(name, []).append(t.transpose(1, 2) if lay else t.squeeze(-1))

    for b0 in range(0, B, chunk):
        sl = slice(b0, min(B, b0 + chunk))
        qc, kc, vc = (t[sl].to(F64).transpose(1, 2) for t in (q, k, v))  # [b, NH, T, H]
        Md = keep[sl].to(F64) * inv_keep if keep is not None else 1.0
        S = ((qc @ kc.transpose(-1, -2)) * s).masked_fill(~vis, float("-inf"))
        m = S.amax(-1, keepdim=True)
        lse = m + torch.log(torch.exp(S - m).sum(-1, keepdim=True))
        P = torch.exp(S - lse)
        Pd = P * Md
        o = Pd @ vc
        Sa = S.masked_fill(~vis, 0.0).abs()
        A = (qc.abs() @ kc.abs().transpose(-1, -2)) * s
        dlt = (cS * A + EXP * (Sa + m.abs()) + EXP).masked_fill(~vis, 0.0)
        dbar = torch.log1p((P * torch.expm1(dlt)).sum(-1, keepdim=True))
        eps = torch.expm1(dlt + dbar)
        F = (1 + sig) * (1 + cT) * (1 + eps) * (1 + r) - 1
        put("o", o)
        put("o_tol", (Pd * F) @ vc.abs() + FLOOR)
        put("lse", lse, False)
        put("lse_tol", dbar + c24 + EXP * (1 + (lse - m).abs()) + 2.0 ** -22 * (m.abs() + lse.abs()) + FLOOR, False)
        if d_o is None:
            continue
        gc = d_o[sl].to(F64).transpose(1, 2)
        dP = gc @ vc.transpose(-1, -2)
        dPd = dP * Md
        D = (Pd * dP).sum(-1, keepdim=True)
        dS = P * (dPd - D) * s
        put("dq", dS @ kc)
        put("dk", dS.transpose(-1, -2) @ qc)
        put("dv", Pd.transpose(-1, -2) @ gc)
        Bg = gc.abs() @ vc.abs().transpose(-1, -2)
        lg = lse_got[sl].to(F64).unsqueeze(-1)
        dlb = cS * A + EXP * (Sa + lse.abs()) + EXP + (lg - lse).abs()
        epb = torch.expm1(dlb).masked_fill(~vis, 0.0)
        e = (cS * Bg + 2.0 ** -23 * dP.abs()) * Md
        if path == "tc":
            og = o_got[sl].to(F64).transpose(1, 2)
            dD = (gc * (og - o)).sum(-1, keepdim=True).abs() + H * U24 * (gc * og).abs().sum(-1, keepdim=True)
        else:
            dD = (P * ((1 + epb) * (1 + c24) * (dPd.abs() + e) - dPd.abs())).sum(-1, keepdim=True)
        E = s * P * (epb * (dPd - D).abs() + (1 + epb) * (e + dD)) * (1 + 2.0 ** -22) + 2.0 ** -22 * dS.abs()
        G = ((1 + r) * (1 + cT) - 1) * dS.abs() + (1 + r) * (1 + cT) * E
        put("dq_tol", G @ kc.abs() + FLOOR)
        put("dk_tol", G.transpose(-1, -2) @ qc.abs() + FLOOR)
        Gv = Pd * ((1 + epb) * (1 + 2.0 ** -23) * (1 + r) * (1 + cT) - 1)
        put("dv_tol", Gv.transpose(-1, -2) @ gc.abs() + FLOOR)
    return {n: torch.cat(ts) for n, ts in out.items()}
