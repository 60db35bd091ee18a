"""CPU oracle for the GritLM embedding hot path — TEST INFRASTRUCTURE ONLY.

A plain-PyTorch (CPU) restatement of the reference algorithm, each function citing the reference
file:line it follows (paths relative to the upstream repo ContextualAI/gritlm @ 9710681).
Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may
import this module; the product path (gritlm_b200/) never does and fails loudly without its CUDA
library.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so this oracle is
pinned against OUTPUTS OF THE REFERENCE ITSELF: `tests/golden/make_golden.py` imports the
reference's own `scripts/modeling_mistral_gritlm.py`, `gritlm/gritlm.py` and
`gritlm/training/model.py` (unmodified) and stores their outputs on seeded inputs in
`tests/golden/*.npz`; `tests/test_oracle_golden.py` checks this file against those fixtures, and
`tests/test_oracle_vs_reference.py` against a second set of inputs (`make_golden_checks.py`).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn.functional as F


@dataclass
class MistralDims:
    hidden_size: int = 4096
    intermediate_size: int = 14336
    num_layers: int = 32
    num_heads: int = 32
    num_kv_heads: int = 8
    head_dim: int = 128
    vocab_size: int = 32000
    rms_eps: float = 1e-5
    rope_theta: float = 10000.0
    max_positions: int = 4096
    num_experts: int = 0          # 0 = dense Mistral MLP; 8 = Mixtral block-sparse MoE
    top_k: int = 2
    router_aux_loss_coef: float = 0.02

    @staticmethod
    def mistral_7b() -> "MistralDims":
        return MistralDims()

    @staticmethod
    def mixtral_8x7b() -> "MistralDims":
        return MistralDims(rope_theta=1e6, num_experts=8, top_k=2, max_positions=4096)

    @staticmethod
    def tiny_moe(num_layers: int = 2, num_experts: int = 8) -> "MistralDims":
        return MistralDims(hidden_size=256, intermediate_size=256, num_layers=num_layers, num_heads=2,
                           num_kv_heads=1, head_dim=128, vocab_size=512, max_positions=512, rope_theta=1e6,
                           num_experts=num_experts, top_k=2)

    @staticmethod
    def tiny(num_layers: int = 2) -> "MistralDims":
        return MistralDims(hidden_size=256, intermediate_size=512, num_layers=num_layers, num_heads=2,
                           num_kv_heads=1, head_dim=128, vocab_size=512, max_positions=512)


def make_weights(dims: MistralDims, seed: int = 1234, dtype=torch.bfloat16, lm_head: bool = True,
                 norm_jitter: float = 0.0, gate_std: float = 0.02) -> Dict[str, torch.Tensor]:
    """HF-style random init (normal(0, 0.02) for Linear/Embedding, RMSNorm weight = 1;
    scripts/modeling_mistral_gritlm.py:819-828) under HF parameter names.  `norm_jitter` perturbs
    the norm weights so that tests also exercise the weight multiply."""
    g = torch.Generator().manual_seed(seed)
    H, I, nh, nkv, dh = dims.hidden_size, dims.intermediate_size, dims.num_heads, dims.num_kv_heads, dims.head_dim

    def lin(o, i):
        return (torch.randn(o, i, generator=g) * 0.02).to(dtype)

    def norm():
        w = torch.ones(H)
        if norm_jitter:
            w = w + norm_jitter * torch.randn(H, generator=g)
        return w.to(dtype)

    sd = {"model.embed_tokens.weight": lin(dims.vocab_size, H)}
    for l in range(dims.num_layers):
        p = f"model.layers.{l}."
        sd[p + "self_attn.q_proj.weight"] = lin(nh * dh, H)
        sd[p + "self_attn.k_proj.weight"] = lin(nkv * dh, H)
        sd[p + "self_attn.v_proj.weight"] = lin(nkv * dh, H)
        sd[p + "self_attn.o_proj.weight"] = lin(H, nh * dh)
        if dims.num_experts:
            # Mixtral names (scripts/modeling_mixtral_gritlm.py:797-837): w1=gate, w3=up, w2=down
            sd[p + "block_sparse_moe.gate.weight"] = (torch.randn(dims.num_experts, H, generator=g) * gate_std).to(dtype)
            for e in range(dims.num_experts):
                q = p + f"block_sparse_moe.experts.{e}."
                sd[q + "w1.weight"] = lin(I, H)
                sd[q + "w2.weight"] = lin(H, I)
                sd[q + "w3.weight"] = lin(I, H)
        else:
            sd[p + "mlp.gate_proj.weight"] = lin(I, H)
            sd[p + "mlp.up_proj.weight"] = lin(I, H)
            sd[p + "mlp.down_proj.weight"] = lin(H, I)
        sd[p + "input_layernorm.weight"] = norm()
        sd[p + "post_attention_layernorm.weight"] = norm()
    sd["model.norm.weight"] = norm()
    if lm_head:
        sd["lm_head.weight"] = lin(dims.vocab_size, H)
    return sd


# ------------------------------------------------------------------------------------------------
# building blocks
# ------------------------------------------------------------------------------------------------
def rms_norm(x: torch.Tensor, weight: torch.Tensor, eps: float) -> torch.Tensor:
    """MistralRMSNorm.forward — scripts/modeling_mistral_gritlm.py:84-89."""
    input_dtype = x.dtype
    h = x.to(torch.float32)
    variance = h.pow(2).mean(-1, keepdim=True)
    h = h * torch.rsqrt(variance + eps)
    return weight * h.to(input_dtype)


def rope_tables(head_dim: int, seq_len: int, base: float, dtype) -> tuple:
    """MistralRotaryEmbedding — modeling_mistral_gritlm.py:93-126: fp32 inv_freq/freqs,
    emb = cat(freqs, freqs), cos/sin cast to the activation dtype at use (:124-125)."""
    inv_freq = 1.0 / (base ** (torch.arange(0, head_dim, 2).float() / head_dim))
    t = torch.arange(seq_len, dtype=inv_freq.dtype)
    freqs = torch.outer(t, inv_freq)
    emb = torch.cat((freqs, freqs), dim=-1)
    return emb.cos().to(dtype), emb.sin().to(dtype)


def rotate_half(x):
    """modeling_mistral_gritlm.py:130-134."""
    x1 = x[..., : x.shape[-1] // 2]
    x2 = x[..., x.shape[-1] // 2:]
    return torch.cat((-x2, x1), dim=-1)


def apply_rope(q, k, cos, sin):
    """apply_rotary_pos_emb — modeling_mistral_gritlm.py:138-163 with position_ids = arange(S)
    (:984-990); q,k are [B, heads, S, dh]."""
    cos = cos[None, None, :, :]
    sin = sin[None, None, :, :]
    return (q * cos) + (rotate_half(q) * sin), (k * cos) + (rotate_half(k) * sin)


def repeat_kv(x, n_rep):
    """modeling_mistral_gritlm.py:182-191."""
    if n_rep == 1:
        return x
    b, h, s, d = x.shape
    return x[:, :, None, :, :].expand(b, h, n_rep, s, d).reshape(b, h * n_rep, s, d)


def additive_mask(attention_mask: Optional[torch.Tensor], B: int, S: int, dtype, is_causal: bool):
    """The 4-D additive mask the reference builds (modeling_mistral_gritlm.py:1005-1036 via
    transformers' _prepare_4d_attention_mask / _prepare_4d_causal_attention_mask): finfo.min on
    padded keys (and on future keys when causal).  Returns None when nothing is masked (the
    sdpa path passes mask=None for all-ones masks)."""
    neg = torch.finfo(dtype).min
    m = None
    if attention_mask is not None and not bool(attention_mask.bool().all()):
        m = torch.zeros(B, 1, S, S, dtype=dtype)
        m = m.masked_fill(attention_mask[:, None, None, :] == 0, neg)
    if is_causal:
        c = torch.full((S, S), neg, dtype=dtype).triu(1)[None, None]
        m = c.expand(B, 1, S, S).clone() if m is None else torch.clamp(m + c, min=neg)
    return m


def attention(q, k, v, mask4d):
    """Eager MistralAttention core — modeling_mistral_gritlm.py:283-310: scores in the activation
    dtype, + additive mask, softmax in fp32 cast back, P·V."""
    dh = q.shape[-1]
    w = torch.matmul(q, k.transpose(2, 3)) / math.sqrt(dh)
    if mask4d is not None:
        w = w + mask4d
    w = F.softmax(w, dim=-1, dtype=torch.float32).to(q.dtype)
    return torch.matmul(w, v)


def decoder_layer(x, sd, prefix, dims: MistralDims, cos, sin, mask4d, router_out=None, kv_out=None, sel_override=None):
    """MistralDecoderLayer.forward — modeling_mistral_gritlm.py:726-785 (attention :627-705,
    MLP :177-178); with dims.num_experts > 0 it is MixtralDecoderLayer (modeling_mixtral_gritlm.py:
    885-962), identical except for the block-sparse MoE in place of the MLP."""
    B, S, H = x.shape
    nh, nkv, dh = dims.num_heads, dims.num_kv_heads, dims.head_dim
    residual = x
    h = rms_norm(x, sd[prefix + "input_layernorm.weight"], dims.rms_eps)
    q = F.linear(h, sd[prefix + "self_attn.q_proj.weight"]).view(B, S, nh, dh).transpose(1, 2)
    k = F.linear(h, sd[prefix + "self_attn.k_proj.weight"]).view(B, S, nkv, dh).transpose(1, 2)
    v = F.linear(h, sd[prefix + "self_attn.v_proj.weight"]).view(B, S, nkv, dh).transpose(1, 2)
    q, k = apply_rope(q, k, cos, sin)
    if kv_out is not None:
        kv_out.append((k, v))  # HF legacy cache entry: post-RoPE keys, values, [B, nkv, S, dh]
    k = repeat_kv(k, nh // nkv)
    v = repeat_kv(v, nh // nkv)
    a = attention(q, k, v, mask4d).transpose(1, 2).contiguous().reshape(B, S, nh * dh)
    x = residual + F.linear(a, sd[prefix + "self_attn.o_proj.weight"])
    residual = x
    h = rms_norm(x, sd[prefix + "post_attention_layernorm.weight"], dims.rms_eps)
    if dims.num_experts:
        y, router_logits = moe_block(h, sd, prefix + "block_sparse_moe.", dims, sel_override)
        if router_out is not None:
            router_out.append(router_logits)
        return residual + y
    g = F.linear(h, sd[prefix + "mlp.gate_proj.weight"])
    u = F.linear(h, sd[prefix + "mlp.up_proj.weight"])
    x = residual + F.linear(F.silu(g) * u, sd[prefix + "mlp.down_proj.weight"])
    return x


def moe_block(h, sd, prefix, dims: MistralDims, sel_override=None):
    """MixtralSparseMoeBlock.forward — scripts/modeling_mixtral_gritlm.py:839-882: router linear in the
    activation dtype, fp32 softmax, top-2, renormalise, cast back, per-expert SwiGLU FFN scaled by the
    routing weight and index_add-ed into a zero tensor of the activation dtype.
    `sel_override` [T, top_k] int64 (tests only) pins the discrete expert choice — e.g. to the decisions the
    device made from its bf16 logits — so that gradients can be compared where a near-tie would otherwise
    send a token to different experts on the two sides; the routing weights are still this function's own."""
    B, S, H = h.shape
    x = h.view(-1, H)
    router_logits = F.linear(x, sd[prefix + "gate.weight"])
    rw = F.softmax(router_logits, dim=1, dtype=torch.float)
    if sel_override is not None:
        sel = sel_override
        rw = rw.gather(1, sel)
    else:
        rw, sel = torch.topk(rw, dims.top_k, dim=-1)
    rw = rw / rw.sum(dim=-1, keepdim=True)
    rw = rw.to(x.dtype)
    out = torch.zeros_like(x)
    mask = F.one_hot(sel, num_classes=dims.num_experts).permute(2, 1, 0)
    for e in range(dims.num_experts):
        idx, top_x = torch.where(mask[e])
        if top_x.shape[0] == 0:
            continue
        cur = x[top_x]
        q = prefix + f"experts.{e}."
        y = F.linear(F.silu(F.linear(cur, sd[q + "w1.weight"])) * F.linear(cur, sd[q + "w3.weight"]), sd[q + "w2.weight"])
        y = y * rw[top_x, idx, None]
        out.index_add_(0, top_x, y.to(x.dtype))
    return out.view(B, S, H), router_logits


def load_balancing_loss(gate_logits, num_experts: int, top_k: int = 2, attention_mask=None):
    """load_balancing_loss_func — scripts/modeling_mixtral_gritlm.py:80-153 (tuple of per-layer
    [B*S, E] router logits)."""
    cat = torch.cat(list(gate_logits), dim=0)
    rw = F.softmax(cat, dim=-1)
    _, sel = torch.topk(rw, top_k, dim=-1)
    emask = F.one_hot(sel, num_experts)
    if attention_mask is None:
        tokens_per_expert = torch.mean(emask.float(), dim=0)
        router_prob = torch.mean(rw, dim=0)
    else:
        b, s = attention_mask.shape
        nl = cat.shape[0] // (b * s)
        am = attention_mask[None, :, :, None, None].expand((nl, b, s, top_k, num_experts)).reshape(-1, top_k, num_experts)
        tokens_per_expert = torch.sum(emask.float() * am, dim=0) / torch.sum(am, dim=0)
        rm = attention_mask[None, :, :, None].expand((nl, b, s, num_experts)).reshape(-1, num_experts)
        router_prob = torch.sum(rw * rm, dim=0) / torch.sum(rm, dim=0)
    return torch.sum(tokens_per_expert * router_prob.unsqueeze(0)) * num_experts


def mistral_forward(*args, **kwargs):
    """No-grad wrapper of `mistral_forward_grad` (inference oracle)."""
    with torch.no_grad():
        return mistral_forward_grad(*args, **kwargs)


def mistral_forward_grad(sd: Dict[str, torch.Tensor], dims: MistralDims, input_ids: torch.Tensor,
                    attention_mask: Optional[torch.Tensor] = None, is_causal: bool = False,
                    dtype=torch.float32, return_layers: bool = False, router_out: Optional[list] = None,
                    kv_out: Optional[list] = None, mask4d_override: Optional[torch.Tensor] = None,
                    routing_override: Optional[list] = None):
    """MistralModel.forward — modeling_mistral_gritlm.py:936-1096 -> last_hidden_state [B,S,H].
    `dtype` is the compute dtype (weights are cast to it): torch.bfloat16 reproduces the
    reference's bf16 rounding points on CPU, torch.float32 is the high-precision oracle.
    Autograd-enabled: pass leaf tensors with requires_grad in `sd` to obtain reference gradients."""
    sd = {k: (v if v.dtype == dtype else v.to(dtype)) for k, v in sd.items()}
    B, S = input_ids.shape
    x = F.embedding(input_ids, sd["model.embed_tokens.weight"])
    cos, sin = rope_tables(dims.head_dim, S, dims.rope_theta, dtype)
    mask4d = additive_mask(attention_mask, B, S, dtype, is_causal)
    if mask4d_override is not None:  # arbitrary visibility pattern (e.g. bidirectional prefix + causal suffix)
        mask4d = mask4d_override.to(dtype)
    layers = []
    for l in range(dims.num_layers):
        x = decoder_layer(x, sd, f"model.layers.{l}.", dims, cos, sin, mask4d, router_out, kv_out,
                          routing_override[l] if routing_override is not None else None)
        if return_layers:
            layers.append(x)
    out = rms_norm(x, sd["model.norm.weight"], dims.rms_eps)
    return (out, layers) if return_layers else out


def lm_logits(sd, hidden):
    """MistralForCausalLM.forward lm_head + .float() — modeling_mistral_gritlm.py:1191-1192."""
    return F.linear(hidden, sd["lm_head.weight"].to(hidden.dtype)).float()


# ------------------------------------------------------------------------------------------------
# pooling / normalise / losses
# ------------------------------------------------------------------------------------------------
def pooling(hidden_state: torch.Tensor, attention_mask: torch.Tensor, method: str, recast: bool = False):
    """GritLM.pooling — gritlm/gritlm.py:178-218 (does NOT mutate the caller's mask)."""
    attention_mask = attention_mask.clone()
    if method == "cls":
        emb = hidden_state[:, 0]
    elif method == "lasttoken":
        b, n, d = hidden_state.size()
        rev = torch.flip(attention_mask, dims=(1,))
        idx = attention_mask.size(1) - torch.argmax(rev, dim=1) - 1
        idx = torch.clamp(idx, min=0)
        gather = idx.unsqueeze(-1).repeat(1, d).unsqueeze(1)
        expanded = attention_mask.unsqueeze(-1).expand((b, n, d)).float()
        emb = torch.gather(hidden_state * expanded, 1, gather).squeeze(dim=1)
    elif method in ("mean", "weightedmean"):
        if method == "weightedmean":
            attention_mask = attention_mask * attention_mask.cumsum(dim=1)
        s = torch.sum(hidden_state * attention_mask.unsqueeze(-1).float(), dim=1)
        d = attention_mask.sum(dim=1, keepdim=True).float()
        emb = s / d
    else:
        raise NotImplementedError(f"Unknown pooling method: {method}")
    return emb.to(hidden_state.dtype) if recast else emb


def normalize(emb: torch.Tensor) -> torch.Tensor:
    """gritlm/gritlm.py:156-158: F.normalize(dim=-1) cast back to the input dtype."""
    return F.normalize(emb, dim=-1).to(emb.dtype)


def encode_tokens(*args, **kwargs):
    with torch.no_grad():
        return encode_tokens_grad(*args, **kwargs)


def encode_tokens_grad(sd, dims, input_ids, attention_mask, pool_mask=None, method="mean", normalized=True,
                       is_causal=False, dtype=torch.float32, routing_override=None):
    """GritLM.encode on pre-tokenised inputs — gritlm/gritlm.py:129-158 (autograd-enabled)."""
    h = mistral_forward_grad(sd, dims, input_ids, attention_mask, is_causal, dtype, routing_override=routing_override)
    pm = attention_mask if pool_mask is None else pool_mask
    if pm is None:
        pm = torch.ones_like(input_ids)
    e = pooling(h, pm, method)
    return normalize(e) if normalized else e


def contrastive_loss(q_reps: torch.Tensor, p_reps: torch.Tensor, temperature: float) -> torch.Tensor:
    """DistributedContrastiveLoss.__call__ on already gathered reps — gritlm/training/model.py:36-47."""
    scores = torch.matmul(q_reps, p_reps.transpose(0, 1)) / temperature
    scores = scores.view(q_reps.size(0), -1)
    target = torch.arange(scores.size(0), dtype=torch.long) * (p_reps.size(0) // q_reps.size(0))
    return F.cross_entropy(scores, target, reduction="mean")


def next_token_loss(labels, logits, vocab_size, loss_gen_type="mixed", loss_gen_factor=1.0):
    """NextTokenLoss.__call__ — gritlm/training/model.py:94-107."""
    shift_logits = logits[..., :-1, :].contiguous().view(-1, vocab_size)
    shift_labels = labels[..., 1:].contiguous().view(-1)
    if loss_gen_type == "token":
        return F.cross_entropy(shift_logits, shift_labels, reduction="sum") / labels.size(0) * loss_gen_factor
    if loss_gen_type == "mixed":
        return F.cross_entropy(shift_logits, shift_labels, reduction="mean") * loss_gen_factor
    raise ValueError(f"Invalid loss_gen_type: {loss_gen_type}")
