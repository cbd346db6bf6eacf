"""The encoder's attention kernels against an fp64 reference, and encoder hidden states row by row.

1. ac_attention (the encoder's own dispatch over caller buffers) against tests/attention_reference.py at every sequence, window
   and padding edge of both kernels, on sharp inputs where every ignored position holds 3e4 (tolerance: TOL_UNITS there).
2. Every valid row of the last hidden state of 1- and 2-layer BERT and ModernBERT models with sharpened attention, through
   the real QKV epilogues (V transpose, RoPE), against an fp64 restatement with the path's fp16 operand rounding.
3. One encoder reused across shapes equals a fresh one bit for bit (stale qk / vT rows from an earlier call are never read).
4. Short sequences (S <= 3) that fill the whole token budget: the transposed-V workspace covers S_pad = 8 > S.
"""
import pytest
import torch

import attention_reference as ar
import modernbert_oracle as mo
from oracle import encoder_oracle as eo

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ 1. the kernels alone
@pytest.mark.parametrize("B,S,heads,kind,window", ar.grid(), ids=lambda v: str(v))
def test_attention_matches_fp64_reference(cabi, B, S, heads, kind, window):
    inp = ar.make_inputs(B, S, heads, kind, window)
    mask = inp["mask"].cuda() if inp["mask"] is not None else None
    ctx = cabi.attention(inp["qk"].cuda(), inp["vT"].cuda(), mask, B, S, heads, window).cpu().double()
    ref, has = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], B, S, heads, window)
    tol = ar.tolerance(inp)
    assert not bool(torch.isnan(ctx).any()), "NaN (or a row never written)"
    assert bool((ctx[~has] == 0).all()), "a row with no visible key must be exactly zero"
    err = (ctx[has] - ref[has]).abs().max().item() if bool(has.any()) else 0.0
    print(f"attention B={B} S={S} heads={heads} {kind} window={window}: max err {err:.3e} = {err / tol:.3f} x tol")
    assert err <= tol, (err, tol)


def test_attention_rejects_bad_arguments(cabi):
    inp = ar.make_inputs(2, 40, 1, "none")
    with pytest.raises(cabi.AdaptiveB200Error):                       # fewer qk rows than B*S
        cabi.attention(inp["qk"][:79].contiguous().cuda(), inp["vT"].cuda(), None, 2, 40, 1, 0)
    with pytest.raises(cabi.AdaptiveB200Error):
        cabi.attention(torch.zeros(1200, 128, dtype=torch.float16, device="cuda"),
                       torch.zeros(2 * 64, 520, dtype=torch.float16, device="cuda"), None, 2, 513, 1, 0)


# ------------------------------------------------------------------------------------------------ 2. hidden states row by row
QK_GAIN = 6.0        # query and key weights x6: random-init scores (std ~0.3 after the 1/8 scale) -> std ~10


def _r16(t):
    return t.to(torch.float16).to(t.dtype)


_MODELS = {}


def _bert(layers):
    key = ("bert", layers)
    if key not in _MODELS:
        sd, cfg, _ = eo.make_bert_state_dict(77, num_hidden_layers=layers, hidden_size=256, num_attention_heads=4,
                                             intermediate_size=512, vocab_size=1000, max_position_embeddings=512)
        for l in range(layers):
            for n in ("query", "key"):
                for wb in ("weight", "bias"):
                    sd[f"encoder.layer.{l}.attention.self.{n}.{wb}"] *= QK_GAIN
        _MODELS[key] = (sd, cfg)
    return _MODELS[key]


# layer types of the two-layer ModernBERT: a sliding layer (window 8) with theta 10 000 and a global one with theta 160 000;
# the one-layer model is layer 0 of it (transformers cannot build a one-layer ModernBertConfig)
MB_OVER = dict(hidden_size=256, num_attention_heads=4, intermediate_size=384, vocab_size=1000, pad_token_id=0, cls_token_id=2,
               sep_token_id=3, bos_token_id=2, eos_token_id=3, local_attention=16, norm_bias=True, attention_bias=True,
               layer_types=["sliding_attention", "full_attention"],
               rope_parameters={"sliding_attention": {"rope_type": "default", "rope_theta": 10000.0},
                                "full_attention": {"rope_type": "default", "rope_theta": 160000.0}})


def _modernbert(layers):
    import types
    key = ("modernbert", layers)
    if key not in _MODELS:
        sd, cfg, _ = mo.make_modernbert_state_dict(78, gamma_noise=0.2, num_hidden_layers=2, **MB_OVER)
        H = cfg.hidden_size
        for l in range(2):
            sd[f"layers.{l}.attn.Wqkv.weight"][:2 * H] *= QK_GAIN
            sd[f"layers.{l}.attn.Wqkv.bias"][:2 * H] *= QK_GAIN
        if layers == 1:
            sd = {k: v for k, v in sd.items() if not k.startswith("layers.1.")}
            d = cfg.to_dict()
            d.update(num_hidden_layers=1, layer_types=cfg.layer_types[:1], sliding_window=cfg.sliding_window)
            cfg = types.SimpleNamespace(**d)
        _MODELS[key] = (sd, cfg)
    return _MODELS[key]


def _bert_encoder(cabi, sd, cfg, max_tokens, cls_only=False):
    return cabi.Encoder(sd, arch="bert", layers=cfg.num_hidden_layers, hidden=cfg.hidden_size, heads=cfg.num_attention_heads,
                        intermediate=cfg.intermediate_size, vocab=cfg.vocab_size, max_pos=cfg.max_position_embeddings,
                        type_vocab=cfg.type_vocab_size, ln_eps=cfg.layer_norm_eps, max_tokens=max_tokens, cls_only=cls_only)


def _encoder(cabi, arch, layers, max_tokens):
    if arch == "bert":
        sd, cfg = _bert(layers)
        return _bert_encoder(cabi, sd, cfg, max_tokens)
    sd, cfg = _modernbert(layers)
    return cabi.Encoder.modernbert(sd, cabi.modernbert_dims(cfg), max_tokens=max_tokens, cls_only=False)


def _ids_mask(arch, B, S, seed):
    ids = (eo.synthetic_ids(B, S, vocab=1000, seed=seed) if arch == "bert" else
           mo.synthetic_ids(B, S, vocab=1000, seed=seed, cls_id=2, sep_id=3))
    mask = torch.ones_like(ids)
    for b in range(1, B, 2):                                   # odd sequences padded: suffix or (every fourth) left padding
        n = max(1, S - 1 - (5 * b) % max(S - 1, 1))
        if b % 4 == 3 and S > 2:
            mask[b, :S - n] = 0
        else:
            mask[b, n:] = 0
    return ids, mask


def _restated_hidden(arch, layers, ids, mask):
    if arch == "bert":
        sd, cfg = _bert(layers)
        sd64 = {k: v.double() for k, v in sd.items()}
        _, h = eo.encoder_forward_cls(sd64, ids, mask, num_heads=cfg.num_attention_heads, ln_eps=cfg.layer_norm_eps,
                                      round_fn=_r16, return_hidden=True)
        return h
    sd, cfg = _modernbert(layers)
    sd64 = {k: v.double() for k, v in sd.items()}
    _, h = mo.modernbert_forward_cls(sd64, ids, mask, cfg, return_hidden=True, round_fn=_r16)
    return h


# Per-row bound on |h - h_ref| / |h_ref| over the valid rows.  The restatement rounds the operands of every product to fp16 as
# the B200 path does, but not always at the same place: P is rounded after, not before, the normalisation, and the BERT path's
# deferred LayerNorm rounds the un-normalised sums and gamma-scaled weights where the restatement rounds LN(y) and W (ModernBERT
# materialises its LayerNorms, so only the first difference remains).  Measured on an NVIDIA B200 (1000 W) over all cases:
# 1.41e-4 (BERT) and 3.0e-5 (ModernBERT); the bounds leave about 3.5x.
HIDDEN_ROW_REL_TOL = {"bert": 5e-4, "modernbert": 1e-4}

HIDDEN_CASES = [(7, 2), (7, 3), (5, 9), (3, 40), (7, 127), (2, 129), (3, 257), (7, 300)]


@pytest.mark.parametrize("arch", ["bert", "modernbert"])
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("B,S", HIDDEN_CASES)
def test_every_valid_hidden_row_matches_the_fp64_restatement(cabi, arch, layers, B, S):
    ids, mask = _ids_mask(arch, B, S, seed=B * 1000 + S)
    enc = _encoder(cabi, arch, layers, B * S)
    enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda())
    got = enc.last_hidden(B, S).cpu().double().view(B, S, -1)
    enc.close()
    want = _restated_hidden(arch, layers, ids, mask)
    keep = mask.bool()
    rel = ((got[keep] - want[keep]).norm(dim=1) / want[keep].norm(dim=1)).max().item()
    tol = HIDDEN_ROW_REL_TOL[arch]
    print(f"hidden {arch} layers={layers} B={B} S={S}: max row rel err {rel:.3e} = {rel / tol:.3f} x tol")
    assert bool(torch.isfinite(got[keep]).all()) and rel < tol, rel


# ------------------------------------------------------------------------------------------------ 3. state across calls
@pytest.mark.parametrize("arch", ["bert", "modernbert"])
def test_a_reused_encoder_equals_a_fresh_one_bit_for_bit(cabi, arch):
    """(7, 300) -> (5, 40) -> (3, 3) -> (7, 300): every call of one encoder equals a freshly created encoder given the same
    input, CLS rows and full hidden state, bit for bit"""
    shapes = [(7, 300), (5, 40), (3, 3), (7, 300)]
    enc = _encoder(cabi, arch, 2, 7 * 300)
    for i, (B, S) in enumerate(shapes):
        ids, mask = _ids_mask(arch, B, S, seed=500 + i)
        ids, mask = ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()
        a = enc.forward_cls(ids, mask).clone()
        ha = enc.last_hidden(B, S)
        fresh = _encoder(cabi, arch, 2, 7 * 300)
        b = fresh.forward_cls(ids, mask)
        hb = fresh.last_hidden(B, S)
        fresh.close()
        assert torch.equal(a, b) and torch.equal(ha, hb), (arch, B, S)
    enc.close()


# ------------------------------------------------------------------------------------------------ 4. S <= 3 at the token budget
@pytest.mark.parametrize("S", [1, 2, 3])
def test_short_sequences_at_the_full_token_budget(cabi, S):
    """max_tokens = 128 * 3 and B = max_tokens / S: B * S_pad (S_pad = 8) is up to 8x max_tokens"""
    sd, cfg, _ = eo.make_bert_state_dict(5, num_hidden_layers=2, hidden_size=256, num_attention_heads=4, intermediate_size=512,
                                         vocab_size=1000)
    max_tokens = 128 * 3
    B = max_tokens // S
    ids = eo.synthetic_ids(B, S, vocab=1000, seed=S)
    mask = torch.ones_like(ids)
    if S > 1:
        mask[1::3, S - 1] = 0
    enc = _bert_encoder(cabi, sd, cfg, max_tokens, cls_only=True)
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    enc.close()
    ref = eo.encoder_forward_cls(sd, ids, mask, num_heads=4, ln_eps=cfg.layer_norm_eps)
    assert (out - ref).norm(dim=1).max().item() < 1e-3


def test_classifier_embeds_a_full_chunk_of_one_word_texts():
    """predict_batch on one-wordpiece texts: [CLS] w [SEP] (S = 3), 21 846 rows = one chunk of 65536 // 3 rows and one more"""
    import tempfile
    import adaptive_classifier_b200 as acb
    from oracle import tiny_bert
    m, cfg = tiny_bert.build()
    clf = acb.AdaptiveClassifier(tiny_bert.save_checkpoint(m, tempfile.mkdtemp(prefix="tiny_bert_s3_")), device="cuda")
    B = 65536 // 3 + 1
    g = torch.Generator().manual_seed(3)
    ids = torch.stack([torch.full((B,), 2), torch.randint(5, len(tiny_bert.VOCAB), (B,), generator=g), torch.full((B,), 3)], 1)
    mask = torch.ones_like(ids)
    out = clf._embed_ids_device(ids.to(torch.int32), mask.to(torch.int32), None).cpu()
    sd = {k: v.detach().float() for k, v in m.state_dict().items()}
    ref = eo.encoder_forward_cls(sd, ids, mask, num_heads=cfg.num_attention_heads, ln_eps=cfg.layer_norm_eps)
    assert out.shape == (B, cfg.hidden_size) and (out - ref).norm(dim=1).max().item() < 1e-3
