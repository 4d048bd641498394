"""Fused runner for the DrakeGPT language models: forward / backward / AdamW / decode
as explicit kernel sequences over preallocated buffers (no autograd tape).

This is the hot path behind ``TransformerLM`` (training step, evaluation and
KV-cached generation) and the generation path of the five smaller models.  One
``Runner`` owns

  * the model's flat parameter arena (``optim.FlatParams``) and, in tensor mode,
    the bf16 weight shadows the tcgen05 GEMMs read;
  * per-(B,T) activation workspaces, allocated once so that the whole step is
    CUDA-graph capturable;
  * the kernel schedule.  Per ResidualBlock2 layer (src/model_component.py:505-506):
        forward   LN1 -> packed-QKV GEMM -> fused causal attention ->
                  proj GEMM (+bias +dropout +residual) -> LN2 ->
                  FFN1 GEMM (+bias +ReLU) -> FFN2 GEMM (+bias +dropout +residual)
        backward  the mirror image: wgrad/dgrad GEMMs fed directly from the
                  row-major activations (MN-major operands), ReLU mask applied in
                  the dgrad epilogue, LN backward fused with the residual-gradient
                  add and the dropout-masked bf16 copy the next GEMM consumes.

Modes: ``"fp32"`` = exact CUDA-core kernels (any model / shape; parity runs),
``"bf16"`` = tcgen05 tensor-core GEMMs with bf16 operands, fp32 accumulation and an
fp32 residual stream (TransformerLM shapes with C % 64 == 0).
"""
import torch

from . import ops
from ._lib import MAJOR_K, MAJOR_MN, KernelError
from .optim import FlatParams, FusedAdamW


def _spec_from_model(model):
    """Describe any of the six LMs as (embeddings, list of block descriptors, head)."""
    kind = type(model).__name__
    names = {id(p): n for n, p in model.named_parameters()}

    def nm(p):
        return None if p is None else names[id(p)]

    spec = {"kind": kind, "tok": nm(model.token_embedding_table.weight), "pos": None, "layers": [], "lm": None,
            "ctx": getattr(model, "context_length", None)}
    if kind == "BigramLM":
        return spec
    spec["pos"] = nm(model.position_embedding_table.weight)
    spec["lm"] = (nm(model.lm_head.weight), nm(model.lm_head.bias))

    def attn_part(m):
        return {"qkv": nm(m.qkv), "NH": m.num_heads, "H": m.head_size, "p_attn": m.attn_dropout}

    if kind in ("SingleHeadAttentionLM", "MultiHeadAttentionLM"):
        d = attn_part(model.sa_head)
        d.update(ln1=None, ln2=None, proj=None, ffn=None, residual=False, p=0.0)
        spec["layers"].append(d)
        return spec
    for blk in model.blocks:
        d = attn_part(blk.sa_head)
        d.update(ln1=None, ln2=None, proj=None, ffn=None, residual=False, p=0.0)
        if hasattr(blk.sa_head, "proj"):
            d["proj"] = (nm(blk.sa_head.proj.weight), nm(blk.sa_head.proj.bias))
            d["residual"] = True
        net = blk.ffwd.net
        if len(net) == 2:
            d["ffn"] = ("relu", nm(net[0].weight), nm(net[0].bias))
        else:
            d["ffn"] = ("mlp", nm(net[0].weight), nm(net[0].bias), nm(net[2].weight), nm(net[2].bias))
        if hasattr(blk, "ln1"):
            d["ln1"] = (nm(blk.ln1.weight), nm(blk.ln1.bias))
            d["ln2"] = (nm(blk.ln2.weight), nm(blk.ln2.bias))
            d["p"] = float(blk.ffwd.net[3].p)
        spec["layers"].append(d)
    return spec


class Runner:
    def __init__(self, model, mode="fp32"):
        if mode not in ("fp32", "bf16"):
            raise ValueError("mode must be 'fp32' or 'bf16'")
        self.model = model
        self.mode = mode
        self.spec = _spec_from_model(model)
        if mode == "bf16":
            ok = self.spec["kind"] == "TransformerLM" and all(
                l["H"] % 8 == 0 and (l["NH"] * l["H"]) % 8 == 0 for l in self.spec["layers"])
            C = model.token_embedding_table.weight.shape[1]
            if not ok or C % 8 != 0:
                raise KernelError("bf16 tensor-core mode needs a TransformerLM with embedding_dim % 8 == 0")
        self.at = torch.float32 if mode == "fp32" else torch.bfloat16
        frozen = ("ln_f.",) if self.spec["kind"] == "TransformerLM" else ()
        self.flat = FlatParams(model, frozen=frozen, with_shadow=(mode == "bf16"))
        self.device = self.flat.device
        self._ws = {}
        self.seed_dev = torch.zeros(1, device=self.device, dtype=torch.int64)
        self.base_seed = 0
        self.opt = None
        self._cache = None
        self._fwd_gen = 0      # bumped by every forward(save=True): the saved activations belong to that call only
        self._flat_gen = 0     # bumped whenever the parameter arena is rebuilt (keys the captured decode graphs)
        self._sm = ops.sm_count()

    # ------------------------------------------------------------------ #
    # plumbing
    # ------------------------------------------------------------------ #
    def _reattach(self):
        if not self.flat.is_attached():
            frozen = ("ln_f.",) if self.spec["kind"] == "TransformerLM" else ()
            old = self.flat
            self.flat = FlatParams(self.model, frozen=frozen, with_shadow=(self.mode == "bf16"))
            if old.p.device == self.flat.p.device and old.n_live == self.flat.n_live:
                self.flat.m.copy_(old.m)
                self.flat.v.copy_(old.v)
            if self.opt is not None:
                self.opt.flat = self.flat
            self.device = self.flat.device
            self._ws = {}
            self._flat_gen += 1
            self.__dict__.pop("_decode_graphs", None)  # captured against the old arena

    def buf(self, key, shape, dtype=None, zero=False):
        dtype = self.at if dtype is None else dtype
        k = (key, tuple(shape), dtype)
        t = self._ws.get(k)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(shape, device=self.device, dtype=dtype)
            self._ws[k] = t
        return t

    def w(self, name):
        """Weight as a GEMM operand: fp32 master (exact mode) or bf16 shadow (tensor mode)."""
        return self.flat.view(name) if self.mode == "fp32" else self.flat.shadow_of(name)

    def f(self, name):
        return None if name is None else self.flat.view(name)

    def g(self, name):
        return self.flat.grad(name)

    def _drop(self, p, site, training):
        if not training or p <= 0.0:
            return None
        return ops.Dropout(p, self.base_seed, site, self.seed_dev)

    def _gemm(self, *a, **k):
        return ops.raw_gemm(*a, **k)

    def _use_relu_mask(self, F):
        return self.mode == "bf16" and F % 64 == 0

    # ------------------------------------------------------------------ #
    # forward
    # ------------------------------------------------------------------ #
    def forward(self, idx, targets=None, training=False, save=False, want_logits=True):
        """Full-sequence forward.  Returns (logits (B*T,V) fp32, loss 0-d tensor or None).

        ``save=True`` keeps every activation the backward pass needs in the
        workspace keyed by layer.
        """
        self._reattach()
        self.flat.refresh_shadow()
        sp = self.spec
        B, T = idx.shape
        M = B * T
        idx = idx.contiguous()
        tok = self.f(sp["tok"])
        V = tok.shape[0]
        if save:
            self._fwd_gen += 1
            self._saved_shape = (B, T)
        if sp["kind"] == "BigramLM":
            logits = self.buf("logits", (M, V), torch.float32)
            ops.raw_embed_fwd(idx, tok, None, logits.view(B, T, V))
        else:
            C = tok.shape[1]
            if sp["ctx"] is not None and T > sp["ctx"]:
                raise KernelError(f"sequence length {T} exceeds context_length {sp['ctx']}")
            x = self.buf("x0", (M, C), torch.float32)
            L0 = sp["layers"][0] if sp["layers"] else None
            fused0 = L0 is not None and L0["ln1"] is not None  # embedding lookup fused with blocks.0.ln1
            if fused0:
                tag = "L0." if save else "tmp."
                a0 = self.buf(tag + "xn1", (M, C))
                ops.raw_embed_ln_fwd(idx, tok, self.f(sp["pos"]), x.view(B, T, C), self.f(L0["ln1"][0]), self.f(L0["ln1"][1]),
                                     a0, self.buf(tag + "mean1", (M,), torch.float32), self.buf(tag + "rstd1", (M,), torch.float32))
            else:
                ops.raw_embed_fwd(idx, tok, self.f(sp["pos"]), x.view(B, T, C))
            ln1_done = fused0
            self._x_last_cast = None
            for li, L in enumerate(sp["layers"]):
                nxt = sp["layers"][li + 1] if li + 1 < len(sp["layers"]) else None
                x, ln1_done = self._layer_fwd(li, L, x, B, T, training, save, ln1_done=ln1_done, nxt=nxt)
            xin = x
            if self._x_last_cast is not None:
                xin = self._x_last_cast  # written by the last block's fused FFN2 kernel
            elif xin.dtype != self.at:
                xin = ops.raw_dropout_scale(x, self.buf("x_last_at", x.shape))
            self._x_last = xin
            Cin = xin.shape[1]
            if self.mode == "bf16" and ops.lmhead_ce_supported(V, Cin) and (targets is not None or want_logits):
                # fused LM head + cross-entropy (src/model.py:599-607): the logits row of every token stays in TMEM;
                # fp32 logits are written only when the caller wants them (the training step does not)
                logits = self.buf("logits", (M, V), torch.float32) if want_logits else None
                loss = dl = None
                if targets is not None:
                    loss = self.buf("loss", (1,), torch.float32)
                    loss.zero_()
                    if save:
                        dl = self.buf("dlogits", (M, (V + 7) // 8 * 8), self.at, zero=True)
                ops.raw_lmhead_ce(xin, self.w(sp["lm"][0]), self.f(sp["lm"][1]),
                                  None if targets is None else targets.contiguous().view(-1), loss, dl, logits)
                return logits, (None if loss is None else loss.view(()))
            logits = self.buf("logits", (M, V), torch.float32)
            self._gemm(xin, self.w(sp["lm"][0]), logits, bias=self.f(sp["lm"][1]))
        loss = None
        if targets is not None:
            loss = self.buf("loss", (1,), torch.float32)
            loss.zero_()
            dl = None
            if save:
                ldl = (V + 7) // 8 * 8
                dl = self.buf("dlogits", (M, ldl), self.at, zero=True)
            ops.raw_cross_entropy(logits, targets.contiguous().view(-1), loss, dl, None, M, V)
            loss = loss.view(())
        return logits, loss

    def _fuse_ln(self, M, N, K):
        """Residual GEMM + the following LayerNorm in one kernel (dgpt_gemm_res_ln): tensor mode, full-row tiles
        (N in {128, 256, 384}) and enough 128-row tiles to occupy the GPU; DGPT_FUSE_LN=0 keeps the two kernels,
        DGPT_FUSE_LN=force fuses at any M (tests)."""
        import os
        env = os.environ.get("DGPT_FUSE_LN", "1")
        return (self.mode == "bf16" and env != "0" and (M >= 64 * self._sm or env == "force")
                and ops.gemm_res_ln_supported(N, K))

    def _layer_fwd(self, li, L, x, B, T, training, save, ln1_done=False, nxt=None):
        """One block; returns (output, whether blocks[li + 1].ln1 has already been applied to it)."""
        M, C = x.shape
        NH, H = L["NH"], L["H"]
        D = NH * H
        tag = (lambda n: f"L{li}.{n}") if save else (lambda n: "tmp." + n)
        ntag = (lambda n: f"L{li + 1}.{n}") if save else (lambda n: "tmp." + n)
        ln2_done = next_ln1_done = False
        if save:
            self._saved_x = getattr(self, "_saved_x", {})
        # ---- attention branch ----
        if L["ln1"] is not None:
            a = self.buf(tag("xn1"), (M, C))
            mean1, rstd1 = self.buf(tag("mean1"), (M,), torch.float32), self.buf(tag("rstd1"), (M,), torch.float32)
            if not ln1_done:
                ops.raw_ln_fwd(x, self.f(L["ln1"][0]), self.f(L["ln1"][1]), a, mean1, rstd1)
        elif x.dtype != self.at:
            a = ops.raw_dropout_scale(x, self.buf(tag("xn1"), (M, C)))
        else:
            a = x
        qkv = self.buf(tag("qkv"), (M, 3 * D))
        self._gemm(a, self.w(L["qkv"]).view(3 * D, C), qkv)
        q3 = qkv.view(B, T, 3 * D)
        att = self.buf(tag("att"), (M, D))
        lse = self.buf(tag("lse"), (B, NH, T), torch.float32)
        ops.raw_attn_fwd(q3[:, :, :D], q3[:, :, D:2 * D], q3[:, :, 2 * D:], att.view(B, T, D), lse, NH, H, H ** -0.5,
                         self._drop(L["p_attn"], 4 * li, training))
        if L["proj"] is not None:
            x1 = self.buf(tag("x1"), (M, C), torch.float32)
            if L["residual"] and L["ffn"] is not None and L["ln2"] is not None and self._fuse_ln(M, C, D):
                # projection + residual + ln2 in one kernel: the fp32 row stays in TMEM for the statistics
                ops.raw_gemm_res_ln(att, self.w(L["proj"][0]), self.f(L["proj"][1]), x, x1, self.f(L["ln2"][0]),
                                    self.f(L["ln2"][1]), self.buf(tag("xn2"), (M, C)),
                                    self.buf(tag("mean2"), (M,), torch.float32), self.buf(tag("rstd2"), (M,), torch.float32),
                                    dropout=self._drop(L["p"], 4 * li + 1, training))
                ln2_done = True
            else:
                self._gemm(att, self.w(L["proj"][0]), x1, bias=self.f(L["proj"][1]),
                           dropout=self._drop(L["p"], 4 * li + 1, training), residual=x if L["residual"] else None)
        else:
            x1 = att
        # ---- feed-forward branch ----
        if L["ffn"] is None:
            out = x1
        else:
            if L["ln2"] is not None:
                b = self.buf(tag("xn2"), (M, C))
                mean2 = self.buf(tag("mean2"), (M,), torch.float32)
                rstd2 = self.buf(tag("rstd2"), (M,), torch.float32)
                if not ln2_done:
                    ops.raw_ln_fwd(x1, self.f(L["ln2"][0]), self.f(L["ln2"][1]), b, mean2, rstd2)
            elif x1.dtype != self.at:
                b = ops.raw_dropout_scale(x1, self.buf(tag("xn2"), (M, C)))
            else:
                b = x1
            if L["ffn"][0] == "relu":
                out = self.buf(tag("x2"), (M, C), torch.float32)
                self._gemm(b, self.w(L["ffn"][1]), out, bias=self.f(L["ffn"][2]), relu=True)
            else:
                F = self.f(L["ffn"][1]).shape[0]
                h = self.buf(tag("h"), (M, F))
                # tensor mode: the GEMM also writes the ReLU bit mask its dgrad twin applies (1/16 of re-reading h)
                hmask = self.buf(tag("hmask"), ((F // 32) * M,), torch.int32) if save and self._use_relu_mask(F) else None
                self._gemm(b, self.w(L["ffn"][1]), h, bias=self.f(L["ffn"][2]), relu=True, relu_mask_out=hmask)
                out = self.buf(tag("x2"), (M, C), torch.float32)
                if L["residual"] and nxt is None and self.at != torch.float32 and self._fuse_ln(M, C, F):
                    # last block: FFN2 + residual, and the bf16 copy the LM head reads, in one kernel
                    self._x_last_cast = self.buf("x_last_at", (M, C))
                    ops.raw_gemm_res_ln(h, self.w(L["ffn"][3]), self.f(L["ffn"][4]), x1, out, None, None,
                                        self._x_last_cast, None, None, dropout=self._drop(L["p"], 4 * li + 2, training))
                elif L["residual"] and nxt is not None and nxt["ln1"] is not None and self._fuse_ln(M, C, F):
                    # FFN2 + residual + the NEXT block's ln1 in one kernel
                    ops.raw_gemm_res_ln(h, self.w(L["ffn"][3]), self.f(L["ffn"][4]), x1, out, self.f(nxt["ln1"][0]),
                                        self.f(nxt["ln1"][1]), self.buf(ntag("xn1"), (M, C)),
                                        self.buf(ntag("mean1"), (M,), torch.float32),
                                        self.buf(ntag("rstd1"), (M,), torch.float32),
                                        dropout=self._drop(L["p"], 4 * li + 2, training))
                    next_ln1_done = True
                else:
                    self._gemm(h, self.w(L["ffn"][3]), out, bias=self.f(L["ffn"][4]),
                               dropout=self._drop(L["p"], 4 * li + 2, training), residual=x1 if L["residual"] else None)
        if save:
            self._saved_x[li] = x
        return out, next_ln1_done

    # ------------------------------------------------------------------ #
    # backward (TransformerLM / ResidualBlock2 structure)
    # ------------------------------------------------------------------ #
    def backward(self, idx, training=True, reducer=None, fwd_gen=None):
        """Backward of the last ``forward(..., save=True)``; gradients are ACCUMULATED into the flat arena.

        The saved activations live in per-shape workspaces shared by every call, so only the LATEST
        ``forward(save=True)`` can be differentiated: ``fwd_gen`` (the value of ``self._fwd_gen`` right after
        the forward the caller wants to differentiate) makes a stale backward raise instead of silently using
        another call's activations.

        ``reducer`` (parallel.GradAllReducer built by ``make_reducer``) is told after the lm_head, after
        every block and after the embeddings that the next gradient bucket is final; in its overlapped mode the
        all-reduce of that slice then runs beside the rest of the backward pass (default: one all-reduce in
        ``reducer.finish()``, see parallel.GradAllReducer).
        """
        sp = self.spec
        if sp["kind"] != "TransformerLM":
            raise KernelError("Runner.backward implements the TransformerLM block structure; smaller models "
                              "train through the autograd Functions in ops.py")
        if fwd_gen is not None and fwd_gen != self._fwd_gen:
            raise KernelError("backward of a stale forward: a later forward(save=True) on this model overwrote the "
                              "saved activations (one forward/backward pair at a time per model; gradient "
                              "accumulation must run forward+backward per micro-batch)")
        B, T = idx.shape
        if getattr(self, "_saved_shape", None) != (B, T):
            raise KernelError(f"backward for a ({B},{T}) batch but the last forward(save=True) saw "
                              f"{getattr(self, '_saved_shape', None)}")
        M = B * T
        tok = self.f(sp["tok"])
        V, C = tok.shape
        sm = self._sm
        dl = self.buf("dlogits", (M, (V + 7) // 8 * 8), self.at, zero=True)
        x_last = self._x_last
        # lm_head: dW = dl^T x, db = colsum(dl), dx = dl W
        tc = self.mode == "bf16"  # tensor mode: bias gradients ride on the wgrad GEMMs (a_colsum)
        self._gemm(dl, x_last, self.g(sp["lm"][0]), a_major=MAJOR_MN, b_major=MAJOR_MN, M=V, N=C, K=M,
                   accumulate=True, split_k=self._splits(V, C, M, sm), a_colsum=self.g(sp["lm"][1]) if tc else None)
        if not tc:
            ops.raw_colsum(dl, self.g(sp["lm"][1]), accumulate=True, M=M, N=V)
        if reducer is not None:
            reducer.bucket_ready()
        gcur = self.buf("g_a", (M, C), torch.float32)
        self._gemm(dl, self.w(sp["lm"][0]), gcur, b_major=MAJOR_MN, M=M, N=C, K=V)
        gm = self.buf("gm", (M, C))
        nl = len(sp["layers"])
        # masked bf16/fp32 copy of the incoming gradient for the last layer's FFN2
        Llast = sp["layers"][-1]
        ops.raw_dropout_scale(gcur, gm, self._drop(Llast["p"], 4 * (nl - 1) + 2, training))
        galt = self.buf("g_b", (M, C), torch.float32)
        for li in range(nl - 1, -1, -1):
            L = sp["layers"][li]
            nxt = sp["layers"][li - 1] if li > 0 else None
            gcur = self._layer_bwd(li, L, nxt, gcur, galt, gm, B, T, training)
            if reducer is not None:
                reducer.bucket_ready()
        # embeddings
        ops.raw_embed_bwd(idx.contiguous(), gcur.view(B, T, C), self.g(sp["tok"]), self.g(sp["pos"]))
        if reducer is not None:
            reducer.bucket_ready()

    def make_reducer(self, group=None):
        """Gradient buckets in the order the backward pass completes them (lm_head, blocks L-1..0, embeddings)."""
        from .parallel import GradAllReducer, PeerAdamW, bucket_ranges
        import os
        import torch.distributed as dist
        # default on the GPUs: ONE kernel for reduce-scatter + AdamW + all-gather over NVLink peer memory;
        # DGPT_DP_MODE=nccl selects the NCCL all-reduce + replicated AdamW schedule (A/B, or no peer access)
        if (self.opt is not None and dist.is_initialized() and dist.get_world_size(group) > 1
                and dist.get_backend(group) == "nccl" and os.environ.get("DGPT_DP_MODE", "peer") == "peer"):
            sp = self.spec
            only_shadow = [sp["lm"][0]] if self.mode == "bf16" else []
            if self.mode == "bf16":
                for L in sp["layers"]:  # the GEMM weights: read through their bf16 shadows only
                    only_shadow += [L["qkv"], L["proj"][0], L["ffn"][1], L["ffn"][3]]
            return PeerAdamW(self.flat, self.opt, group, shadow_only=only_shadow)
        nl = len(self.spec["layers"])
        groups = [("lm_head.",)] + [(f"blocks.{i}.",) for i in range(nl - 1, -1, -1)]
        groups.append(("token_embedding_table.", "position_embedding_table."))
        red = GradAllReducer(self.flat.g, bucket_ranges(self.flat.slots, self.flat.n_live, groups), group)
        if self.opt is not None:
            self.opt.grad_scale = red.grad_scale
        return red

    @staticmethod
    def _splits(n_out_rows, n_out_cols, k, sm, colsum=False):
        # column tile of the wgrad GEMM: 192 for N = 192 / 384 / 576 / 960, 256 for a wide output with few row tiles that
        # also carries a column sum (FFN2: 384 x 1536), else 128 (launch_gemm_tc picks the same)
        bn = 192 if (n_out_cols % 192 == 0 and n_out_cols % 256 != 0 and n_out_cols < 1024 and n_out_rows >= 1024) else 128
        if colsum and n_out_cols % 256 == 0 and n_out_cols >= 512 and n_out_rows < 1024:
            bn = 256
        tiles = ((n_out_rows + 127) // 128) * ((n_out_cols + bn - 1) // bn)
        return max(1, min(sm // max(tiles, 1), k // 512))

    def _layer_bwd(self, li, L, nxt, g, g_other, gm, B, T, training):
        """g: dL/dx_out (fp32), gm: dropout-masked copy of g in the activation dtype.  Returns dL/dx_in."""
        M, C = g.shape
        NH, H = L["NH"], L["H"]
        D = NH * H
        sm = self._sm
        tag = lambda n: f"L{li}.{n}"  # noqa: E731
        at = self.at
        F = self.f(L["ffn"][1]).shape[0]
        x_in = self._saved_x[li]
        xn1, qkv, att = self.buf(tag("xn1"), (M, C)), self.buf(tag("qkv"), (M, 3 * D)), self.buf(tag("att"), (M, D))
        lse = self.buf(tag("lse"), (B, NH, T), torch.float32)
        x1, xn2, h = self.buf(tag("x1"), (M, C), torch.float32), self.buf(tag("xn2"), (M, C)), self.buf(tag("h"), (M, F))
        mean1, rstd1 = self.buf(tag("mean1"), (M,), torch.float32), self.buf(tag("rstd1"), (M,), torch.float32)
        mean2, rstd2 = self.buf(tag("mean2"), (M,), torch.float32), self.buf(tag("rstd2"), (M,), torch.float32)
        # ---- FFN2: y = h W2^T + b2 (dropout, residual) ----
        tc = self.mode == "bf16"  # tensor mode: every bias gradient is a by-product of its wgrad GEMM
        self._gemm(gm, h, self.g(L["ffn"][3]), a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True,
                   split_k=self._splits(C, F, M, sm, colsum=tc), a_colsum=self.g(L["ffn"][4]) if tc else None)
        if not tc and li == len(self.spec["layers"]) - 1:  # other layers: fused into the LN1 backward of layer li+1
            ops.raw_colsum(gm, self.g(L["ffn"][4]), accumulate=True)
        dh = self.buf("dh", (M, F))
        if self._use_relu_mask(F):
            self._gemm(gm, self.w(L["ffn"][3]), dh, b_major=MAJOR_MN,
                       relu_mask_in=self.buf(tag("hmask"), ((F // 32) * M,), torch.int32))
        else:
            self._gemm(gm, self.w(L["ffn"][3]), dh, b_major=MAJOR_MN, relu_aux=h)
        # ---- FFN1: h = relu(xn2 W1^T + b1) ----
        self._gemm(dh, xn2, self.g(L["ffn"][1]), a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True,
                   split_k=self._splits(F, C, M, sm), a_colsum=self.g(L["ffn"][2]) if tc else None)
        if not tc:
            ops.raw_colsum(dh, self.g(L["ffn"][2]), accumulate=True)
        dxn = self.buf("dxn", (M, C))  # activation dtype: bf16 in tensor mode halves this round trip
        self._gemm(dh, self.w(L["ffn"][1]), dxn, b_major=MAJOR_MN)
        # ---- LN2 backward + residual-gradient add + masked copy for the proj GEMMs ----
        g1 = g_other
        ops.raw_ln_bwd(dxn, x1, self.f(L["ln2"][0]), mean2, rstd2, g, g1, self.g(L["ln2"][0]), self.g(L["ln2"][1]),
                       dxm=gm, dropout=self._drop(L["p"], 4 * li + 1, training),
                       dxm_colsum=None if tc else self.g(L["proj"][1]))
        # ---- proj: y = att Wp^T + bp (dropout, residual) ----
        self._gemm(gm, att, self.g(L["proj"][0]), a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True,
                   split_k=self._splits(C, D, M, sm), a_colsum=self.g(L["proj"][1]) if tc else None)
        datt = self.buf("datt", (M, D))
        self._gemm(gm, self.w(L["proj"][0]), datt, b_major=MAJOR_MN)
        # ---- attention ----
        dqkv = self.buf("dqkv", (M, 3 * D))
        q3, d3 = qkv.view(B, T, 3 * D), dqkv.view(B, T, 3 * D)
        q, k, v = q3[:, :, :D], q3[:, :, D:2 * D], q3[:, :, 2 * D:]
        a3, g3 = att.view(B, T, D), datt.view(B, T, D)
        dq, dk, dv = d3[:, :, :D], d3[:, :, D:2 * D], d3[:, :, 2 * D:]
        nbytes = ops.attn_bwd_scratch_bytes(q, k, v, a3, lse, g3, dq, dk, dv, NH, H)
        scratch = self.buf("attn_scratch", ((nbytes + 3) // 4,), torch.float32)
        ops.raw_attn_bwd(q, k, v, a3, lse, g3, dq, dk, dv, scratch, NH, H, H ** -0.5,
                         self._drop(L["p_attn"], 4 * li, training))
        # ---- QKV projection ----
        self._gemm(dqkv, xn1, self.g(L["qkv"]).view(3 * D, C), a_major=MAJOR_MN, b_major=MAJOR_MN, accumulate=True,
                   split_k=self._splits(3 * D, C, M, sm))
        self._gemm(dqkv, self.w(L["qkv"]).view(3 * D, C), dxn, b_major=MAJOR_MN)
        # ---- LN1 backward + residual add (+ masked copy for the previous layer's FFN2) ----
        g0 = g
        ops.raw_ln_bwd(dxn, x_in, self.f(L["ln1"][0]), mean1, rstd1, g1, g0, self.g(L["ln1"][0]),
                       self.g(L["ln1"][1]), dxm=gm if nxt is not None else None,
                       dropout=self._drop(nxt["p"], 4 * (li - 1) + 2, training) if nxt is not None else None,
                       dxm_colsum=self.g(nxt["ffn"][4]) if (nxt is not None and not tc) else None)
        return g0

    # ------------------------------------------------------------------ #
    # training step
    # ------------------------------------------------------------------ #
    def configure_optimizer(self, lr, betas=(0.9, 0.95), eps=1e-8, weight_decay=1e-2):
        self._reattach()
        self.flat.attach_grads()  # p.grad become views of the flat gradient arena
        self.opt = FusedAdamW(self.flat, lr, betas, eps, weight_decay)
        return self.opt

    def train_step_launch(self, idx, targets, reducer=None):
        """Enqueue forward + backward (+ bucketed DP all-reduce) + AdamW; returns the loss tensor.

        Gradients are expected to be zero on entry (the fused AdamW clears them).
        Everything is enqueued on the current stream and is CUDA-graph capturable.
        """
        if self.opt is None:
            raise KernelError("call configure_optimizer() first")
        _, loss = self.forward(idx, targets, training=True, save=True, want_logits=False)
        self.backward(idx, training=True, reducer=reducer)
        if reducer is not None and getattr(reducer, "fused_optimizer", False):
            reducer.launch_update()  # gradient reduction, AdamW and the parameter all-gather in one kernel
        else:
            if reducer is not None:
                reducer.finish()
            self.opt.launch(zero_grad=True)
        ops.raw_counter_add(self.seed_dev, 1)
        return loss

    def train_step(self, idx, targets, reducer=None):
        self.opt.upload()
        loss = self.train_step_launch(idx, targets, reducer)
        self.opt.t += 1
        return loss

    # ------------------------------------------------------------------ #
    # generation: KV-cached while the window has not slid, full-window
    # recompute afterwards (reference semantics, src/model.py:611-636)
    # ------------------------------------------------------------------ #
    def _decode_token(self, tok_ids, t, caches):
        """One new token per sequence at absolute position ``t``; returns the final hidden state (B,C)."""
        sp = self.spec
        Bn = tok_ids.shape[0]
        tok = self.f(sp["tok"])
        C = tok.shape[1]
        x = self.buf("d.x0", (Bn, C), torch.float32)
        ops.raw_embed_fwd(tok_ids.view(Bn, 1), tok, self.f(sp["pos"]), x.view(Bn, 1, C), pos_offset=t)
        for li, L in enumerate(sp["layers"]):
            NH, H = L["NH"], L["H"]
            D = NH * H
            # [B, ctx, 3D] sequence-major: the packed q | k | v of position t is written by the QKV GEMM through a
            # strided output view (row pitch ctx * 3D), and the keys / values of one sequence sit next to each other,
            # 3D elements apart, so the decode attention streams whole DRAM pages instead of one 128-byte row per page
            cache = caches[li]
            if L["ln1"] is not None:
                a = self.buf("d.xn1", (Bn, C))
                ops.raw_ln_fwd(x, self.f(L["ln1"][0]), self.f(L["ln1"][1]), a, self.buf("d.mean", (Bn,), torch.float32),
                               self.buf("d.rstd", (Bn,), torch.float32))
            elif x.dtype != self.at:
                a = ops.raw_dropout_scale(x, self.buf("d.xn1", (Bn, C)))
            else:
                a = x
            self._gemm(a, self.w(L["qkv"]).view(3 * D, C), cache[:, t])
            q = cache[:, t:t + 1, :D]
            kv = cache[:, : t + 1]  # (B, t+1, 3D) view
            att = self.buf("d.att", (Bn, D))
            if ops.decode_attn_supported(q, kv, H):  # tensor mode, head size 64: the KV-streaming decode kernel
                ops.raw_decode_attn(q, kv[:, :, D:2 * D], kv[:, :, 2 * D:], att.view(Bn, 1, D), NH, H, H ** -0.5)
            else:
                ops.raw_attn_fwd(q, kv[:, :, D:2 * D], kv[:, :, 2 * D:], att.view(Bn, 1, D), None, NH, H, H ** -0.5)
            if L["proj"] is not None:
                x1 = self.buf("d.x1", (Bn, C), torch.float32)
                self._gemm(att, self.w(L["proj"][0]), x1, bias=self.f(L["proj"][1]),
                           residual=x if L["residual"] else None)
            else:
                x1 = att
            if L["ffn"] is None:
                x = x1
                continue
            if L["ln2"] is not None:
                b = self.buf("d.xn2", (Bn, C))
                ops.raw_ln_fwd(x1, self.f(L["ln2"][0]), self.f(L["ln2"][1]), b,
                               self.buf("d.mean", (Bn,), torch.float32), self.buf("d.rstd", (Bn,), torch.float32))
            elif x1.dtype != self.at:
                b = ops.raw_dropout_scale(x1, self.buf("d.xn2", (Bn, C)))
            else:
                b = x1
            out = self.buf(f"d.x2.{li & 1}", (Bn, C), torch.float32)
            if L["ffn"][0] == "relu":
                self._gemm(b, self.w(L["ffn"][1]), out, bias=self.f(L["ffn"][2]), relu=True)
            else:
                h = self.buf("d.h", (Bn, self.f(L["ffn"][1]).shape[0]))
                self._gemm(b, self.w(L["ffn"][1]), h, bias=self.f(L["ffn"][2]), relu=True)
                self._gemm(h, self.w(L["ffn"][3]), out, bias=self.f(L["ffn"][4]),
                           residual=x1 if L["residual"] else None)
            x = out
        return x

    def _persistent_decode_ok(self, Bn):
        """The one-launch persistent decoder covers the TransformerLM block structure in tensor mode, head size 64,
        context <= 256.  It is used while every sequence gets a 16-CTA cluster of its own (<= 4 sequences: 134 us per
        token against 187-191 us for the per-position graphs); with two sequences per cluster (5-8) it measures 216 us
        against 191-193 us, so those batches take the graph path.  DGPT_DECODE_PERSISTENT=0 turns it off,
        DGPT_DECODE_PERSISTENT=force uses it up to the kernel's limit of 8 sequences (A/B runs, tests).
        The shape limits (width, layers, context, cluster budget) are the kernel's own, dgpt_decode_persistent_supported:
        a model outside them takes the per-position path."""
        import os
        from . import _lib
        sp = self.spec
        env = os.environ.get("DGPT_DECODE_PERSISTENT", "1")
        if self.mode != "bf16" or env == "0":
            return False
        limit = int(_lib.lib().dgpt_decode_persistent_max_batch())
        if not (1 <= Bn <= (limit if env == "force" else min(limit, 4))):
            return False
        if sp["ctx"] is None or not sp["layers"]:
            return False
        V, C = self.f(sp["tok"]).shape
        for L in sp["layers"]:
            if (L["ln1"] is None or L["ln2"] is None or L["proj"] is None or not L["residual"]
                    or L["ffn"] is None or L["ffn"][0] != "mlp" or L["NH"] * L["H"] != C):
                return False
        # the kernel takes one (NH, H, F) for every layer
        L0 = sp["layers"][0]
        F = self.f(L0["ffn"][1]).shape[0]
        if any((L["NH"], L["H"], self.f(L["ffn"][1]).shape[0]) != (L0["NH"], L0["H"], F) for L in sp["layers"]):
            return False
        return ops.decode_persistent_supported(Bn, len(sp["layers"]), C, L0["NH"], L0["H"], F, V, sp["ctx"])

    def _decode_persistent(self, seqw, caches, Bn, t_begin, t_end, t_sample, greedy, seed_dev, sampling=None):
        import ctypes as C_
        from . import _lib
        sp = self.spec
        tok = self.f(sp["tok"])
        V, C = tok.shape
        L0 = sp["layers"][0]
        NH, H = L0["NH"], L0["H"]
        F = self.f(L0["ffn"][1]).shape[0]
        lib = _lib.lib()
        nfl = int(lib.dgpt_decode_persistent_scratch_floats(Bn, C, NH, F, V))
        scratch = self.buf("d.pscratch", (nfl,), torch.float32)
        ptrs = (C_.c_void_p * (12 * len(sp["layers"])))()
        for li, L in enumerate(sp["layers"]):
            ts = [self.w(L["qkv"]), self.w(L["proj"][0]), self.w(L["ffn"][1]), self.w(L["ffn"][3]),
                  self.f(L["ln1"][0]), self.f(L["ln1"][1]), self.f(L["ln2"][0]), self.f(L["ln2"][1]),
                  self.f(L["proj"][1]), self.f(L["ffn"][2]), self.f(L["ffn"][4]), caches[li]]
            for j, t in enumerate(ts):
                ptrs[12 * li + j] = t.data_ptr()
        _lib.check(lib.dgpt_decode_persistent_ex(ptrs, len(sp["layers"]), tok.data_ptr(), self.f(sp["pos"]).data_ptr(),
                                                 self.w(sp["lm"][0]).data_ptr(), self.f(sp["lm"][1]).data_ptr(),
                                                 seqw.data_ptr(), scratch.data_ptr(), Bn, C, NH, H, F, V, sp["ctx"],
                                                 int(t_begin), int(t_end), int(t_sample), int(bool(greedy)), 0,
                                                 seed_dev.data_ptr(), ops._p(sampling), 0, ops._stream()),
                   "dgpt_decode_persistent_ex")

    @torch.no_grad()
    def generate(self, idx, max_new_tokens, greedy=False, seed=None, use_graphs=None, temperature=1.0, top_k=None,
                 top_p=1.0):
        """(B,t0) int64 -> (B,t0+N) int64.  Sampling (softmax -> multinomial, or argmax) runs on the device, with
        optional temperature, top-k and top-p (nucleus) cut-offs (rule: warp_sample_row in csrc/sample.cuh; the
        defaults draw exactly the plain multinomial).  The settings live in a device buffer beside the sampling seed,
        so one captured graph serves every setting.

        While the window has not slid (t < context_length) every position is one KV-cached decode step.
        Tensor mode, up to 8 sequences: ONE cooperative launch of the persistent decoder (``dgpt_decode_persistent``)
        walks all in-window positions.  Larger batches: per-position kernel sequences (tcgen05 GEMMs on the M = batch
        rows + the KV-streaming attention kernel), each (batch, position) step captured once in a CUDA graph with
        ``use_graphs`` (default: tensor mode) -- the sequence buffer, KV caches and sampling seed live in device memory.
        After the slide every token is a full-window recompute (reference semantics, src/model.py:625).
        """
        ops.check_sampling(temperature, top_k, top_p)
        self._reattach()
        self.flat.refresh_shadow()
        sp = self.spec
        Bn, t0 = idx.shape
        total = t0 + max_new_tokens
        seed = ops.next_seed() if seed is None else int(seed)
        tok = self.f(sp["tok"])
        V = tok.shape[0]
        sampling = self.buf("d.sampling", (3,), torch.int32)
        settings = (float(temperature), top_k, float(top_p))
        prev = self.__dict__.get("_sampling_in_buf")
        if prev is None or prev[0] is not sampling or prev[1] != settings:  # upload on change only: a host copy syncs
            sampling.copy_(ops.sampling_settings(temperature, top_k, top_p))
            self._sampling_in_buf = (sampling, settings)
        if sp["kind"] == "BigramLM":
            seq = torch.empty((total, Bn), device=self.device, dtype=torch.int64)  # time-major
            seq[:t0].copy_(idx.t())
            logits = self.buf("d.logits", (Bn, V), torch.float32)
            for t in range(t0 - 1, total - 1):
                ops.raw_embed_fwd(seq[t].view(Bn, 1), tok, None, logits.view(Bn, 1, V))
                ops.raw_sample(logits, seq[t + 1], 0, greedy, seed, t, sampling=sampling)
            return seq.t().contiguous()
        ctx = sp["ctx"]
        if use_graphs is None:
            use_graphs = self.mode == "bf16"
        # the in-window part of the sequence lives in a persistent buffer so captured graphs stay valid
        win_len = min(total, ctx + 1)
        seqw = self.buf("d.seq", (ctx + 1, Bn), torch.int64)
        seq = seqw if total <= ctx + 1 else torch.empty((total, Bn), device=self.device, dtype=torch.int64)
        seq[:t0].copy_(idx.t())
        if seq is not seqw:
            seqw[:min(t0, ctx + 1)].copy_(seq[:min(t0, ctx + 1)])
        caches = [self.buf(f"d.cache{li}", (Bn, ctx, 3 * L["NH"] * L["H"])) for li, L in enumerate(sp["layers"])]
        logits = self.buf("d.logits", (Bn, V), torch.float32)
        sample_seed = self.buf("d.seed", (1,), torch.int64)
        sample_seed.fill_(seed)
        graphs = self.__dict__.setdefault("_decode_graphs", {})
        n_in = min(total - 1, ctx)  # positions decoded inside the window
        if self._persistent_decode_ok(Bn) and n_in > 0:
            # small batch: ONE launch (a thread-block cluster per sequence) walks every in-window position (all layers, KV append, attention,
            # LM head, sampling) -- no per-token launches at all
            self._decode_persistent(seqw, caches, Bn, 0, n_in, t0 - 1, greedy, sample_seed, sampling)
            n_done = n_in
        else:
            n_done = 0

        def step_kernels(t, draw, greedy_flag):
            x = self._decode_token(seqw[t], t, caches)
            if draw:
                xin = x if x.dtype == self.at else ops.raw_dropout_scale(x, self.buf("d.xl", x.shape))
                self._gemm(xin, self.w(sp["lm"][0]), logits, bias=self.f(sp["lm"][1]))
                ops.raw_sample(logits, seqw[t + 1], 0, greedy_flag, 0, t, seed_dev=sample_seed, sampling=sampling)

        for t in range(n_done, n_in):
            draw = t >= t0 - 1
            if not use_graphs:
                step_kernels(t, draw, greedy)
                continue
            key = (Bn, t, draw, bool(greedy), self._flat_gen)
            g = graphs.get(key)
            if g is None:
                step_kernels(t, draw, greedy)  # warm-up: allocates workspaces, loads kernels
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    step_kernels(t, draw, greedy)
                graphs[key] = g
            else:
                g.replay()
        if seq is not seqw:
            seq[:win_len].copy_(seqw[:win_len])
        for t in range(ctx, total - 1):
            if t >= t0 - 1:
                # window slid: absolute positions of every token change -> recompute the window (reference
                # semantics, src/model.py:625: idx[:, -context_length:])
                win = seq[t - ctx + 1: t + 1].t().contiguous()
                full, _ = self.forward(win)
                last = full.view(Bn, ctx, V)[:, -1, :]
                ops.raw_sample(last, seq[t + 1], 0, greedy, seed, t, sampling=sampling)
        return seq[:total].t().contiguous()
