"""ORACLE (test infrastructure only -- never imported by the product path).

CPU fp32 restatement of the ModernBERT encoder (HF `transformers` 5.5.0 `models/modernbert/modeling_modernbert.py`) as the
reference's `_get_embeddings` uses it (classifier.py:1271-1275: last_hidden_state[:, 0] -> F.normalize):

    embeddings   LayerNorm(tok_embeddings[ids])                                           :52-71
    block        x = x + Wo(attn(attn_norm(x)));  x = x + mlp(mlp_norm(x))  (pre-LN)        :313-343
                 attn_norm is the identity in layer 0
    attention    fused Wqkv [3H, H] viewed as (3, heads, 64); RoPE on q and k with the rotate_half convention
                 (pairs d and d + 32), inv_freq = 1 / theta^(2i/64) in fp32, positions arange(S), scale 64^-0.5;
                 sliding layers see keys with |q - k| <= sliding_window (inclusive, masking_utils.py:121-131)
    mlp          input, gate = Wi(x).chunk(2);  Wo(gelu_erf(input) * gate)                 :74-91
    output       final_norm(x)

`layer_types`, the per-type rope theta, the window and the three bias switches are taken from the config as given.
Pinned against HF ModernBertModel (eager and sdpa) by tests/test_modernbert_cpu.py.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional, Tuple

import torch

Tensor = torch.Tensor


def _ln(x: Tensor, sd: Dict[str, Tensor], name: str, eps: float) -> Tensor:
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    y = (x - mu) / torch.sqrt(var + eps) * sd[name + ".weight"]
    b = sd.get(name + ".bias")
    return y + b if b is not None else y


def _lin(x: Tensor, sd: Dict[str, Tensor], name: str, r: Callable[[Tensor], Tensor] = lambda t: t) -> Tensor:
    y = r(x) @ r(sd[name + ".weight"]).t()
    b = sd.get(name + ".bias")
    return y + b if b is not None else y


def _gelu_erf(x: Tensor) -> Tensor:
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def layer_windows_thetas(cfg) -> Tuple[List[int], List[float]]:
    """per layer: key window (0 = global attention) and rope theta, as the config states them"""
    wins, thetas = [], []
    for t in cfg.layer_types:
        wins.append(int(cfg.sliding_window) if t == "sliding_attention" else 0)
        thetas.append(float(cfg.rope_parameters[t]["rope_theta"]))
    return wins, thetas


def rope_cos_sin(theta: float, S: int, dim: int = 64) -> Tuple[Tensor, Tensor]:
    """cos, sin [S, dim] exactly as HF computes them (fp32 inv_freq, fp32 angles)"""
    inv_freq = 1.0 / (theta ** (torch.arange(0, dim, 2, dtype=torch.int64).to(dtype=torch.float) / dim))
    freqs = torch.arange(S, dtype=torch.float32)[:, None] * inv_freq[None, :]
    emb = torch.cat((freqs, freqs), dim=-1)
    return emb.cos(), emb.sin()


def _rotate_half(x: Tensor) -> Tensor:
    h = x.shape[-1] // 2
    return torch.cat((-x[..., h:], x[..., :h]), dim=-1)


def modernbert_forward_cls(sd: Dict[str, Tensor], ids: Tensor, mask, cfg, return_hidden: bool = False,
                           inclusive_window: bool = True, round_fn: Optional[Callable[[Tensor], Tensor]] = None):
    """unit-norm CLS rows fp32 [B, H] (and the final-normed hidden state [B, S, H] with return_hidden).
    inclusive_window=False restates the off-by-one variant |q - k| < window (only to show that tests can see it).
    round_fn (as in oracle/encoder_oracle.py) is applied to both operands of every matrix product -- the linears, q k^T after
    RoPE and P V with the normalised P -- to restate the B200 path's fp16 operand rounding."""
    r = round_fn if round_fn is not None else (lambda t: t)
    B, S = ids.shape
    if mask is None:
        mask = torch.ones_like(ids)
    eps = float(cfg.norm_eps)
    H = cfg.hidden_size
    nh = cfg.num_attention_heads
    dh = H // nh
    x = _ln(sd["embeddings.tok_embeddings.weight"][ids], sd, "embeddings.norm", eps)
    wins, thetas = layer_windows_thetas(cfg)
    keep = mask.to(torch.bool)[:, None, None, :]                   # [B, 1, 1, S]
    dist = (torch.arange(S)[:, None] - torch.arange(S)[None, :]).abs()
    neg = torch.finfo(torch.float32).min
    for l in range(cfg.num_hidden_layers):
        p = f"layers.{l}."
        h = x if l == 0 else _ln(x, sd, p + "attn_norm", eps)
        qkv = _lin(h, sd, p + "attn.Wqkv", r).view(B, S, 3, nh, dh)
        q, k, v = (qkv[:, :, j].transpose(1, 2) for j in range(3))  # [B, nh, S, dh]
        cos, sin = rope_cos_sin(thetas[l], S, dh)
        q = q * cos + _rotate_half(q) * sin
        k = k * cos + _rotate_half(k) * sin
        vis = keep
        if wins[l]:
            near = (dist <= wins[l]) if inclusive_window else (dist < wins[l])
            vis = vis & near[None, None]
        scores = (r(q) @ r(k).transpose(-1, -2)) * dh ** -0.5
        scores = scores.masked_fill(~vis, neg)
        ctx = r(torch.softmax(scores, dim=-1)) @ r(v)
        ctx = ctx.transpose(1, 2).reshape(B, S, H)
        x = x + _lin(ctx, sd, p + "attn.Wo", r)
        h = _ln(x, sd, p + "mlp_norm", eps)
        a, g = _lin(h, sd, p + "mlp.Wi", r).chunk(2, dim=-1)
        x = x + _lin(_gelu_erf(a) * g, sd, p + "mlp.Wo", r)
    x = _ln(x, sd, "final_norm", eps)
    cls = x[:, 0, :]
    unit = cls / cls.norm(dim=1, keepdim=True).clamp_min(1e-12)
    if return_hidden:
        return unit, x
    return unit


def make_modernbert_state_dict(seed: int = 1234, gamma_noise: float = 0.0, bias_shift: float = 0.0, **cfg_over):
    """Seeded random-init ModernBERT (base architecture unless overridden): torch.manual_seed(seed); ModernBertModel(cfg).
    gamma_noise > 0 draws non-unit LayerNorm weights (and non-zero biases where norm_bias) from the same seed;
    bias_shift adds a constant to the attn.Wo / mlp.Wo biases, which pushes the residual stream's row mean up.
    Returns (state_dict, config, model) with the model carrying the same parameters."""
    from transformers import ModernBertConfig, ModernBertModel

    torch.manual_seed(seed)
    cfg = ModernBertConfig(**cfg_over)
    m = ModernBertModel(cfg)
    m.eval()
    with torch.no_grad():
        g = torch.Generator().manual_seed(seed + 1)
        for name, t in m.named_parameters():
            if gamma_noise and "norm" in name:
                if name.endswith(".weight"):
                    t.copy_(1.0 + gamma_noise * torch.randn(t.shape, generator=g))
                else:
                    t.copy_(gamma_noise * torch.randn(t.shape, generator=g))
            if bias_shift and name.endswith(("attn.Wo.bias", "mlp.Wo.bias")):
                t.add_(bias_shift)
    sd = {k: v.detach().clone().float() for k, v in m.state_dict().items()}
    return sd, cfg, m


def synthetic_ids(B: int, S: int, vocab: int = 50368, seed: int = 7, cls_id: int = 50281, sep_id: int = 50282) -> Tensor:
    """uniform in [1000, vocab), CLS first, SEP last, int64 [B, S]"""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(min(1000, vocab // 2), vocab, (B, S), generator=g, dtype=torch.int64)
    ids[:, 0] = min(cls_id, vocab - 1)
    ids[:, -1] = min(sep_id, vocab - 1)
    return ids
