"""The tiny seeded BERT checkpoint the reference ran on in golden_classifier.npz and golden_training.npz (test infrastructure).

Its float32 weights (1.26 MB) are rebuilt from the seeds below instead of being stored; each fixture keeps the SHA-256 of the
state dict it was recorded with (`bert_sha256`), and `model()` refuses a rebuild with another digest: a torch or transformers
release that initialises BertModel differently fails here, not as a parity mismatch further on.
"""
from __future__ import annotations

import hashlib

import numpy as np
import torch

WORDS = [f"w{i}" for i in range(195)]
VOCAB = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + WORDS


def build(hidden: int = 128):
    """seeded 2-layer BERT over VOCAB -> (BertModel, BertConfig)"""
    from transformers import BertConfig, BertModel
    cfg = BertConfig(vocab_size=len(VOCAB), hidden_size=hidden, num_hidden_layers=2, num_attention_heads=2,
                     intermediate_size=2 * hidden, max_position_embeddings=64, type_vocab_size=2, pad_token_id=0)
    torch.manual_seed(1234)
    model = BertModel(cfg)
    g = torch.Generator().manual_seed(99)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if "LayerNorm" in n or n.endswith(".bias"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
            elif "weight" in n and p.dim() == 2:
                # word embeddings x4: token identity survives to the CLS row, so the classes are learnable (nearest-centroid
                # accuracy 0.93 on the sentences of oracle/make_golden.py) and the loops do not early-stop at once
                p.mul_(4.0 if "word_embeddings" in n else 3.0)
        # ... and the constant part of the CLS row's input ([CLS] word row, position 0, token types) is zeroed, otherwise every
        # sentence embeds within 0.2 of every other one and 10 epochs of lr 1e-3 learn nothing (mean pair distance 1.14 now)
        model.embeddings.word_embeddings.weight[2].zero_()
        model.embeddings.position_embeddings.weight[0].zero_()
        model.embeddings.token_type_embeddings.weight.zero_()
    return model, cfg


def digest(state_dict) -> str:
    """SHA-256 over name, dtype, shape and bytes of every entry (torch tensors or numpy arrays), in name order"""
    h = hashlib.sha256()
    for name in sorted(state_dict):
        v = state_dict[name]
        a = np.ascontiguousarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v)
        h.update(f"{name}|{a.dtype.str}|{a.shape}|".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def model(expected_digest: str):
    """build() checked against the digest a fixture recorded"""
    m, cfg = build()
    got = digest(m.state_dict())
    if got != str(expected_digest):
        raise RuntimeError(f"the seeded tiny BERT no longer reproduces the checkpoint of the fixture (sha256 {got}, "
                           f"recorded {expected_digest}): this torch / transformers initialises BertModel differently")
    return m, cfg


def save_checkpoint(m, path: str) -> str:
    """model + tokenizer over VOCAB as a from_pretrained() directory"""
    from transformers import BertTokenizerFast
    m.save_pretrained(path)
    # transformers 5.x: BertTokenizerFast(vocab_file=...) silently keeps only the special tokens (every word -> [UNK]);
    # the vocabulary has to be passed as a dict
    BertTokenizerFast(vocab={w: i for i, w in enumerate(VOCAB)}, do_lower_case=True).save_pretrained(path)
    return path
