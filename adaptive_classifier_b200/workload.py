"""Synthetic workloads of BASELINE.json / SURVEY.md section 8(d), shared by bench.py, __graft_entry__.smoke() and tests.

No network, no datasets, no checkpoints: seeded random-init bert-base (and ModernBERT-base) architecture, synthetic token ids,
class-structured synthetic prototype rows (row j belongs to class j mod C)."""
from __future__ import annotations

import torch


def bert_base_state_dict(seed: int = 1234, **cfg_over):
    """HF BertModel(BertConfig()) == bert-base-uncased architecture, random init under torch.manual_seed(seed)."""
    from transformers import BertConfig, BertModel
    torch.manual_seed(seed)
    cfg = BertConfig(**cfg_over)
    m = BertModel(cfg, add_pooling_layer=False)
    m.eval()
    return m, cfg


def modernbert_base_state_dict(seed: int = 1234, **cfg_over):
    """HF ModernBertModel(ModernBertConfig()) == ModernBERT-base architecture (22 layers, H 768, I 1152, vocab 50368),
    random init under torch.manual_seed(seed)."""
    from transformers import ModernBertConfig, ModernBertModel
    torch.manual_seed(seed)
    cfg = ModernBertConfig(**cfg_over)
    m = ModernBertModel(cfg)
    m.eval()
    return m, cfg


def modernbert_synthetic_ids(B: int, S: int, vocab: int = 50368, seed: int = 7) -> torch.Tensor:
    """uniform in [1000, vocab), CLS = 50281 first, SEP = 50282 last, no padding; int32 [B,S] on the host."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(min(1000, vocab - 1), vocab, (B, S), generator=g, dtype=torch.int64)
    ids[:, 0] = min(50281, vocab - 1)
    ids[:, -1] = min(50282, vocab - 1)
    return ids.to(torch.int32)


def synthetic_ids(B: int, S: int, vocab: int = 30522, seed: int = 7) -> torch.Tensor:
    """uniform in [1000, vocab), [CLS]=101 first, [SEP]=102 last, no padding; int32 [B,S] on the host."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(min(1000, vocab - 1), vocab, (B, S), generator=g, dtype=torch.int64)
    ids[:, 0] = min(101, vocab - 1)
    ids[:, -1] = min(102, vocab - 1)
    return ids.to(torch.int32)


def class_centres(C: int, D: int, device="cpu") -> torch.Tensor:
    g = torch.Generator().manual_seed(0)
    return torch.nn.functional.normalize(torch.randn(C, D, generator=g), dim=1).to(device)


def synthetic_rows(lo: int, hi: int, D: int, C: int, seed: int, device="cuda", chunk: int = 131072) -> torch.Tensor:
    """rows [lo,hi) of the synthetic index: normalize(centre[j mod C] + 0.5*randn/sqrt(D)); generated on `device` in chunks
    with a device generator seeded by (seed, GLOBAL chunk start): any row range of the same index has the same bits, so a row
    shard equals the corresponding slice of the unsharded matrix (the N > 1 parity check of bench.py relies on it)."""
    cen = class_centres(C, D, device)
    out = torch.empty((hi - lo, D), dtype=torch.float32, device=device)
    for s in range(lo - lo % chunk, hi, chunk):
        g = torch.Generator(device=device).manual_seed(seed * 1_000_003 + s)
        noise = torch.randn((chunk, D), generator=g, device=device) * (0.5 / D ** 0.5)
        a, e = max(s, lo), min(hi, s + chunk)
        j = torch.arange(a, e, device=device) % C
        out[a - lo : e - lo] = torch.nn.functional.normalize(cen[j] + noise[a - s : e - s], dim=1)
    return out


def synthetic_queries_embeddings(B: int, D: int, C: int, seed: int = 1, device="cuda") -> torch.Tensor:
    """isolated-kNN queries: same construction around the same centres, query b belongs to class b mod C."""
    cen = class_centres(C, D, device)
    g = torch.Generator(device=device).manual_seed(seed + 777)
    noise = torch.randn((B, D), generator=g, device=device) * (0.5 / D ** 0.5)
    return torch.nn.functional.normalize(cen[torch.arange(B, device=device) % C] + noise, dim=1)
