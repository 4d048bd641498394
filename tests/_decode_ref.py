"""fp64 restatement of the KV-cached decoders (csrc/decode.cu and Runner._decode_token).  Test infrastructure only.

The kernels read bf16 shadows of the matrix weights, so those are rounded to bf16 first; everything else is fp64.
Values are rounded to bf16 exactly where the path under test stores bf16:
  * persistent decoder (``graph=False``): the k | v of the KV cache (q is read back in fp32, the activations stay in
    fp32 shared memory);
  * per-position path (``graph=True``): also q, the LayerNorm outputs and the attention output (bf16 GEMM / attention
    inputs), the FFN hidden activation and the last hidden state the LM head reads.
With the tokens the kernel actually wrote (teacher forcing), the KV-cached decode is one causal forward over them."""
import torch

F64 = torch.float64


def bf16(x):
    return x.to(torch.bfloat16).to(F64)


def weights_from_state_dict(sd):
    """The decoder's operands from a TransformerLM state_dict (reference names): packed q | k | v rows per layer."""
    nl = len([k for k in sd if k.endswith("heads.0.key.weight")])
    nh = len([k for k in sd if k.startswith("blocks.0.") and k.endswith("key.weight")])
    layers = []
    for i in range(nl):
        b = f"blocks.{i}."
        qkv = [sd[f"{b}sa_head.heads.{j}.{n}.weight"] for n in ("query", "key", "value") for j in range(nh)]
        layers.append(dict(wqkv=torch.cat(qkv), wproj=sd[b + "sa_head.proj.weight"], bproj=sd[b + "sa_head.proj.bias"],
                           w1=sd[b + "ffwd.net.0.weight"], b1=sd[b + "ffwd.net.0.bias"],
                           w2=sd[b + "ffwd.net.2.weight"], b2=sd[b + "ffwd.net.2.bias"],
                           ln1g=sd[b + "ln1.weight"], ln1b=sd[b + "ln1.bias"],
                           ln2g=sd[b + "ln2.weight"], ln2b=sd[b + "ln2.bias"]))
    return dict(tok=sd["token_embedding_table.weight"], pos=sd["position_embedding_table.weight"],
                wlm=sd["lm_head.weight"], blm=sd["lm_head.bias"], NH=nh, layers=layers)


def _ln(x, g, b):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * g.to(F64) + b.to(F64)


def reference(W, seq, t1, graph=False):
    """seq: [>= t1, B] time-major token ids.  Returns (rows, logits): rows[l] = [B, t1, 3D] q | k | v of layer l at
    every position (before the cache's bf16 store), logits = [B, t1, V] (the logits drawn from at position t)."""
    H = 64
    NH = W["NH"]
    D = NH * H
    ids = seq[:t1].t().cpu()
    B = ids.shape[0]
    r = bf16 if graph else (lambda v: v)
    x = W["tok"].to(F64)[ids] + W["pos"].to(F64)[:t1]
    mask = torch.ones(t1, t1, dtype=torch.bool).tril()
    rows = []
    for L in W["layers"]:
        qkv = r(_ln(x, L["ln1g"], L["ln1b"])) @ bf16(L["wqkv"]).t()
        rows.append(qkv)
        q = r(qkv[..., :D]).view(B, t1, NH, H).transpose(1, 2)
        k = bf16(qkv[..., D:2 * D]).view(B, t1, NH, H).transpose(1, 2)
        v = bf16(qkv[..., 2 * D:]).view(B, t1, NH, H).transpose(1, 2)
        s = (q @ k.transpose(-1, -2)) * H ** -0.5
        p = torch.softmax(s.masked_fill(~mask, float("-inf")), -1)
        att = r((p @ v).transpose(1, 2).reshape(B, t1, D))
        x = x + att @ bf16(L["wproj"]).t() + L["bproj"].to(F64)
        h = r(torch.relu(r(_ln(x, L["ln2g"], L["ln2b"])) @ bf16(L["w1"]).t() + L["b1"].to(F64)))
        x = x + h @ bf16(L["w2"]).t() + L["b2"].to(F64)
    logits = r(x) @ bf16(W["wlm"]).t() + W["blm"].to(F64)
    return rows, logits
