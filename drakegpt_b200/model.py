"""Drop-in counterparts of the reference's ``src/model.py`` language models.

``BigramLM``, ``SingleHeadAttentionLM``, ``MultiHeadAttentionLM``, ``BlocksLM``,
``ResidualBlocksLM`` and ``TransformerLM`` keep the reference constructor
signatures, ``forward(idx, targets=None) -> (logits, loss)`` return shapes
(logits are (B*T, V) when targets are given, SURVEY Q6), ``generate(idx,
max_new_tokens)`` and the ``state_dict`` layout of the shipped ``model/*.pt``.

Execution:
  * ``forward`` of the five small models (and of ``TransformerLM`` in fp32 mode)
    composes the exact-path autograd Functions of ``ops.py``;
  * ``TransformerLM`` in bf16 mode runs the fused tensor-core ``engine.Runner``
    (also reachable as ``model.runner()`` for the graph-captured training step);
  * ``generate`` always runs the Runner: KV-cached decode with on-device sampling
    until the context window slides, full-window recompute afterwards.  ``greedy=True``
    (argmax) is an extension used by the parity tests (SURVEY Q13); so are ``temperature``,
    ``top_k`` and ``top_p``, whose defaults keep the reference's plain multinomial.
"""
from collections import OrderedDict

import torch
import torch.nn as nn

from . import ops
from .engine import Runner
from .model_component import Block, Head, MultiHeadAttention, ResidualBlock, ResidualBlock2


def model_params(params: dict, model_type: str, vocab_size: int):
    """The reference's parameter-count *estimate* printed by train.py (src/model.py:8-63).

    It is not the real count (SURVEY Q14: 11 223 632 vs 10 800 464 actual for the scaled
    TransformerLM); kept so that the CLI prints the same number.  ``count_parameters`` is exact.
    """
    C, T, L = params["embedding_dim"], params["context_length"], params["num_layers"]
    est = OrderedDict()
    est["embedding/position"] = C * T
    est["embedding/character"] = C * vocab_size
    est["attention/kqv"] = 3 * C * C
    est["attention"] = C + est["attention/kqv"] + C * C
    est["mlp/ffw"] = 4 * C * C
    est["mlp"] = C + 2 * est["mlp/ffw"]
    est["blocks"] = (est["attention"] + est["mlp"]) * L
    est["lmhead/ffw"] = C * vocab_size
    total = est["embedding/character"]
    if model_type != "BigramLM":
        total += est["embedding/position"] + est["attention/kqv"] + est["lmhead/ffw"]
    if model_type in ("SingleHeadAttentionLM", "MultiHeadAttentionLM"):
        total += est["embedding/position"] + est["lmhead/ffw"]
    if model_type == "BlocksLM":
        total += (est["attention/kqv"] + est["mlp/ffw"]) * L
    if model_type == "ResidualBlocksLM":
        total += (est["attention/kqv"] + 2 * est["mlp/ffw"]) * L
    if model_type == "TransformerLM":
        total += est["blocks"] + vocab_size
    return total


def count_parameters(model):
    return sum(p.numel() for p in model.parameters())


class _RunnerLoss(torch.autograd.Function):
    """Autograd bridge for the fused Runner: lets ``loss.backward()`` drive the engine's backward."""

    @staticmethod
    def forward(ctx, runner, idx, targets, training, *params):
        logits, loss = runner.forward(idx, targets, training=training, save=True)
        ctx.runner, ctx.training, ctx.idx, ctx.fwd_gen = runner, training, idx, runner._fwd_gen
        ctx.names = [n for n, _ in runner.model.named_parameters()]
        ctx.mark_non_differentiable(logits)
        return logits.clone(), loss.clone()

    @staticmethod
    def backward(ctx, _dlogits, dloss):
        r = ctx.runner
        keep = r.flat.g.clone()
        r.flat.g.zero_()
        r.backward(ctx.idx, training=ctx.training, fwd_gen=ctx.fwd_gen)
        fresh = r.flat.g * dloss
        r.flat.g.copy_(keep)
        grads = []
        for n in ctx.names:
            o, k, shp = r.flat.slots[n]
            grads.append(None if n in r.flat.frozen_names else fresh[o:o + k].view(shp))
        return (None, None, None, None, *grads)


class _LM(nn.Module):
    """Shared plumbing: device checks, loss/logit shaping, Runner-backed generation."""

    _mode = "fp32"

    def _check(self, idx):
        if not idx.is_cuda:
            raise ops._lib.KernelError("drakegpt_b200 models run on CUDA tensors only (no CPU fallback); "
                                       "move the model and inputs to a B200 with .to('cuda')")

    def runner(self):
        r = self.__dict__.get("_runner")
        if r is None or r.mode != self._mode:
            r = Runner(self, self._mode)
            self.__dict__["_runner"] = r
        return r

    def _finish(self, logits, targets):
        """logits (B,T,V) -> reference return convention (src/model.py:601-609)."""
        if targets is None:
            return logits, None
        B, T, V = logits.shape
        flat = logits.view(B * T, V)
        return flat, ops.cross_entropy(flat, targets.view(B * T))

    @torch.no_grad()
    def generate(self, idx, max_new_tokens, greedy=False, seed=None, temperature=1.0, top_k=None, top_p=1.0):
        """Continue ``idx`` (B, t0) by ``max_new_tokens`` tokens.  ``temperature`` (> 0) divides the logits, ``top_k``
        (None or >= 1) keeps the k most likely tokens (ties at the k-th logit kept), ``top_p`` (in (0, 1]) keeps the
        smallest most-likely prefix whose mass reaches it.  The defaults are the reference's softmax -> multinomial;
        ``greedy=True`` (argmax) ignores them.  ``seed`` fixes the draw."""
        ops.check_sampling(temperature, top_k, top_p)
        self._check(idx)
        return self.runner().generate(idx, max_new_tokens, greedy=greedy, seed=seed, temperature=temperature,
                                      top_k=top_k, top_p=top_p)


class BigramLM(_LM):
    """logits = Embedding(V,V)[idx] (src/model.py:65-130)."""

    def __init__(self, vocab_size):
        super().__init__()
        self.token_embedding_table = nn.Embedding(vocab_size, vocab_size)

    def forward(self, idx, targets=None):
        self._check(idx)
        return self._finish(ops.embed(idx, self.token_embedding_table.weight), targets)


class SingleHeadAttentionLM(_LM):
    """tok+pos embedding -> one Head -> lm_head (src/model.py:133-227)."""

    def __init__(self, vocab_size, embedding_dim, context_length, head_size):
        super().__init__()
        self.context_length = context_length
        self.token_embedding_table = nn.Embedding(vocab_size, embedding_dim)
        self.position_embedding_table = nn.Embedding(context_length, embedding_dim)
        self.sa_head = Head(head_size, embedding_dim, context_length)
        self.lm_head = nn.Linear(embedding_dim, vocab_size)

    def _body(self, x):
        return self.sa_head(x)

    def forward(self, idx, targets=None):
        self._check(idx)
        if idx.shape[1] > self.context_length:
            raise IndexError(f"sequence length {idx.shape[1]} exceeds context_length {self.context_length}")
        x = ops.embed(idx, self.token_embedding_table.weight, self.position_embedding_table.weight)
        x = self._body(x)
        return self._finish(ops.linear(x, self.lm_head.weight, self.lm_head.bias), targets)


class MultiHeadAttentionLM(SingleHeadAttentionLM):
    """... -> MultiHeadAttention(num_heads, head_size // num_heads) -> lm_head (src/model.py:230-331)."""

    def __init__(self, vocab_size, embedding_dim, context_length, head_size, num_heads):
        _LM.__init__(self)
        self.context_length = context_length
        self.token_embedding_table = nn.Embedding(vocab_size, embedding_dim)
        self.position_embedding_table = nn.Embedding(context_length, embedding_dim)
        self.sa_head = MultiHeadAttention(num_heads, head_size // num_heads, embedding_dim, context_length)
        self.lm_head = nn.Linear(embedding_dim, vocab_size)


class BlocksLM(SingleHeadAttentionLM):
    """... -> num_layers x Block -> lm_head (src/model.py:334-432)."""

    _block = staticmethod(lambda C, T, NH: Block(C, T, NH))

    def __init__(self, vocab_size, embedding_dim, context_length, num_heads, num_layers):
        _LM.__init__(self)
        self.context_length = context_length
        self.token_embedding_table = nn.Embedding(vocab_size, embedding_dim)
        self.position_embedding_table = nn.Embedding(context_length, embedding_dim)
        self.blocks = nn.Sequential(*[self._block(embedding_dim, context_length, num_heads) for _ in range(num_layers)])
        self.lm_head = nn.Linear(embedding_dim, vocab_size)

    def _body(self, x):
        return self.blocks(x)


class ResidualBlocksLM(BlocksLM):
    """... -> num_layers x ResidualBlock -> lm_head (src/model.py:435-533)."""

    _block = staticmethod(lambda C, T, NH: ResidualBlock(C, NH, T))


class TransformerLM(_LM):
    """Pre-LN transformer with dropout (src/model.py:535-636).

    ``ln_f`` exists (checkpoint key, parameter) but is never applied, exactly like the
    reference (SURVEY Q1).  ``precision``: "auto" picks the bf16 tensor-core engine when
    the shape can feed tcgen05 tiles (embedding_dim % 64 == 0, head size % 16 == 0,
    embedding_dim >= 128), else the exact fp32 path; "fp32" / "bf16" force one.
    """

    def __init__(self, vocab_size, embedding_dim, context_length, num_heads, num_layers, dropout, precision="auto"):
        super().__init__()
        self.context_length = context_length
        self.token_embedding_table = nn.Embedding(vocab_size, embedding_dim)
        self.position_embedding_table = nn.Embedding(context_length, embedding_dim)
        self.blocks = nn.Sequential(
            *[ResidualBlock2(embedding_dim, num_heads, context_length, dropout) for _ in range(num_layers)])
        self.ln_f = nn.LayerNorm(embedding_dim)
        self.lm_head = nn.Linear(embedding_dim, vocab_size)
        if precision == "auto":
            hs = embedding_dim // num_heads
            precision = "bf16" if (embedding_dim % 64 == 0 and embedding_dim >= 128 and hs % 16 == 0) else "fp32"
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'auto', 'fp32' or 'bf16'")
        self._mode = precision

    @property
    def precision(self):
        return self._mode

    def set_precision(self, precision):
        self._mode = precision
        return self

    def forward(self, idx, targets=None):
        self._check(idx)
        B, T = idx.shape
        if T > self.context_length:
            raise IndexError(f"sequence length {T} exceeds context_length {self.context_length}")
        if self._mode == "fp32":
            x = ops.embed(idx, self.token_embedding_table.weight, self.position_embedding_table.weight)
            x = self.blocks(x)
            return self._finish(ops.linear(x, self.lm_head.weight, self.lm_head.bias), targets)
        r = self.runner()
        if targets is None or not torch.is_grad_enabled():
            if self.training:
                r.base_seed = ops.next_seed()
            logits, loss = r.forward(idx, targets, training=self.training)
            logits = logits.clone()
            return (logits.view(B, T, -1), None) if targets is None else (logits, loss.clone())
        r.base_seed = ops.next_seed()
        return _RunnerLoss.apply(r, idx, targets, self.training, *self.parameters())
