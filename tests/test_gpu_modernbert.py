"""ModernBERT on the B200 path (ac_encoder_create_modernbert): every case against the fp32 oracle
(tests/modernbert_oracle.py, pinned against HF ModernBertModel by tests/test_modernbert_cpu.py).

Tolerances are those of the BERT encoder: unit CLS rows within 1e-3 (L2), squared distances to 2048 seeded unit prototypes
within 1e-3, unit norm within 1e-5."""
import tempfile
import types

import numpy as np
import pytest
import torch

import modernbert_oracle as mo

pytestmark = pytest.mark.gpu

BASE = dict()                                                  # ModernBertConfig defaults = ModernBERT-base
LARGE = dict(hidden_size=1024, num_attention_heads=16, intermediate_size=2624)
SMALL_WINDOW = dict(norm_bias=True, attention_bias=True, mlp_bias=True, local_attention=16,
                    layer_types=["sliding_attention", "full_attention", "sliding_attention"],
                    rope_parameters={"sliding_attention": {"rope_type": "default", "rope_theta": 500.0},
                                     "full_attention": {"rope_type": "default", "rope_theta": 20000.0}})

_MODELS = {}


def _model(layers, over, seed=11, bias_shift=0.0):
    key = (layers, repr(sorted(over.items())), seed, bias_shift)
    if key not in _MODELS:
        _MODELS.clear()                                        # one model at a time (22-layer base is 600 MB of fp32)
        if layers == 1:
            # transformers 5.5.0 cannot build a one-layer ModernBertConfig (a single layer type makes it read rope_parameters
            # as one flat entry and then reject it): take layer 0 of a two-layer model and describe it with a plain namespace
            sd, cfg, m = mo.make_modernbert_state_dict(seed, gamma_noise=0.2, bias_shift=bias_shift, num_hidden_layers=2, **over)
            sd = {k: v for k, v in sd.items() if not k.startswith("layers.1.")}
            d = cfg.to_dict()
            d.update(num_hidden_layers=1, layer_types=cfg.layer_types[:1])
            _MODELS[key] = (sd, types.SimpleNamespace(**d), None)
        else:
            _MODELS[key] = mo.make_modernbert_state_dict(seed, gamma_noise=0.2, bias_shift=bias_shift,
                                                         num_hidden_layers=layers, **over)
    return _MODELS[key]


def _encoder(cabi, sd, cfg, max_tokens, cls_only=True):
    return cabi.Encoder.modernbert(sd, cabi.modernbert_dims(cfg), max_tokens=max_tokens, cls_only=cls_only)


def _ids_mask(B, S, vocab, pad, seed=7):
    ids = mo.synthetic_ids(B, S, vocab=vocab, seed=seed)
    mask = torch.ones_like(ids)
    if pad:
        g = torch.Generator().manual_seed(seed + 1)
        for b in range(1, B, 2):
            n = int(torch.randint(2, S, (1,), generator=g))
            mask[b, n:] = 0
    return ids, mask


def _check(got, want, what=""):
    got, want = got.double().cpu(), want.double()
    dq = (got - want).norm(dim=1).max().item()
    P = torch.nn.functional.normalize(torch.randn(2048, got.shape[1], generator=torch.Generator().manual_seed(5),
                                                  dtype=torch.float64), dim=1)
    dd = (torch.cdist(got, P) ** 2 - torch.cdist(want, P) ** 2).abs().max().item()
    nrm = (got.norm(dim=1) - 1).abs().max().item()
    assert dq < 1e-3 and dd < 1e-3 and nrm < 1e-5, (what, dq, dd, nrm)
    return dq, dd


@pytest.mark.parametrize("layers, S, pad, over", [
    (1, 40, True, BASE), (1, 512, False, BASE),
    (3, 40, True, BASE), (3, 128, False, BASE), (3, 300, True, BASE), (3, 512, True, BASE),
    (3, 40, True, SMALL_WINDOW), (3, 300, True, SMALL_WINDOW),
    (22, 128, True, BASE), (22, 300, True, BASE),
])
def test_unit_cls_rows_match_the_oracle(cabi, layers, S, pad, over):
    sd, cfg, _ = _model(layers, over)
    B = 6
    ids, mask = _ids_mask(B, S, cfg.vocab_size, pad)
    enc = _encoder(cabi, sd, cfg, B * S)
    got = enc.forward_cls(ids.to(torch.int32).cuda(), mask.cuda())
    _check(got, mo.modernbert_forward_cls(sd, ids, mask, cfg), (layers, S, pad))


def test_large_shape_covers_the_geglu_tail(cabi):
    """H 1024, 16 heads, 2I = 5248: the last 256-column tile of Wi is half empty"""
    sd, cfg, _ = _model(4, LARGE)
    ids, mask = _ids_mask(4, 128, cfg.vocab_size, True)
    for cls_only in (True, False):
        enc = _encoder(cabi, sd, cfg, 4 * 128, cls_only=cls_only)
        _check(enc.forward_cls(ids.to(torch.int32).cuda(), mask.cuda()), mo.modernbert_forward_cls(sd, ids, mask, cfg))


def test_biases_on_with_a_large_residual_mean(cabi):
    """norm / attention / mlp biases on and +3 on every attn.Wo / mlp.Wo bias: the pre-LN residual stream's row mean grows
    with depth, which is where a deferred (folded) LayerNorm would cancel"""
    over = dict(norm_bias=True, attention_bias=True, mlp_bias=True)
    sd, cfg, _ = _model(6, over, bias_shift=3.0)
    ids, mask = _ids_mask(4, 128, cfg.vocab_size, True)
    enc = _encoder(cabi, sd, cfg, 4 * 128)
    _check(enc.forward_cls(ids.to(torch.int32).cuda(), mask.cuda()), mo.modernbert_forward_cls(sd, ids, mask, cfg))


def test_full_hidden_state_equals_hf_last_hidden_state(cabi):
    sd, cfg, hf = _model(3, BASE)
    B, S = 4, 300
    ids, mask = _ids_mask(B, S, cfg.vocab_size, True)
    full = _encoder(cabi, sd, cfg, B * S, cls_only=False)
    u_full = full.forward_cls(ids.to(torch.int32).cuda(), mask.cuda())
    hid = full.last_hidden(B, S).view(B, S, -1).cpu()
    with torch.no_grad():
        ref = hf(input_ids=ids, attention_mask=mask).last_hidden_state
    v = mask.bool()
    rel = ((hid - ref)[v].norm(dim=1) / ref[v].norm(dim=1)).max().item()
    assert rel < 2e-3, rel
    cls = _encoder(cabi, sd, cfg, B * S, cls_only=True)
    u_cls = cls.forward_cls(ids.to(torch.int32).cuda(), mask.cuda())
    assert (u_full - u_cls).abs().max().item() < 1e-4


def test_benched_batch_sampled_rows(cabi):
    """B = 512 x S = 128, ModernBERT-base at 22 layers (the shape tools/bench_modernbert.py times)"""
    sd, cfg, _ = _model(22, BASE, seed=1234)
    B, S = 512, 128
    ids = mo.synthetic_ids(B, S, vocab=cfg.vocab_size)
    enc = _encoder(cabi, sd, cfg, B * S)
    got = enc.forward_cls(ids.to(torch.int32).cuda())
    rows = torch.tensor([0, 1, 77, 200, 255, 256, 400, 511])
    _check(got[rows.cuda()], mo.modernbert_forward_cls(sd, ids[rows], None, cfg))


def test_type_ids_are_ignored(cabi):
    sd, cfg, _ = _model(1, BASE)
    ids, mask = _ids_mask(3, 40, cfg.vocab_size, True)
    enc = _encoder(cabi, sd, cfg, 3 * 40)
    a = enc.forward_cls(ids.to(torch.int32).cuda(), mask.cuda()).clone()
    b = enc.forward_cls(ids.to(torch.int32).cuda(), mask.cuda(), type_ids=torch.ones_like(ids).cuda())
    assert torch.equal(a, b)


def test_pipeline_host_graph_step_equals_the_eager_step(cabi):
    sd, cfg, _ = _model(3, SMALL_WINDOW)
    B, S, k, C, N = 8, 40, 5, 7, 3000
    enc = _encoder(cabi, sd, cfg, B * S)
    P = torch.nn.functional.normalize(torch.randn(N, cfg.hidden_size, generator=torch.Generator().manual_seed(2)), dim=1).cuda()
    row_class = (torch.arange(N) % C).to(torch.int32).cuda()
    pl = cabi.Pipeline(enc, P, B, S, k, row_class=row_class)
    for rep in range(4):                                       # eager, capture, replay, replay
        ids = mo.synthetic_ids(B, S, vocab=cfg.vocab_size, seed=50 + rep).to(torch.int32)
        oc_h, osc_h = pl.predict_host(ids.pin_memory())
        oc_h, osc_h = oc_h.clone(), osc_h.clone()
        oc, osc = pl.predict_device(ids.cuda())
        assert torch.equal(oc.cpu(), oc_h) and torch.equal(osc.cpu(), osc_h), rep
    emb, _, _ = pl.debug_views(B)
    _check(emb, mo.modernbert_forward_cls(sd, ids.long(), None, cfg))
    pl.close()


def test_unsupported_configs_raise_before_any_device_allocation(cabi):
    from transformers import ModernBertConfig, ModernBertModel
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    for over in (dict(hidden_activation="gelu_pytorch_tanh"), dict(hidden_size=704, num_attention_heads=11),
                 dict(intermediate_size=1000), dict(hidden_size=768, num_attention_heads=6)):
        m = ModernBertModel(ModernBertConfig(num_hidden_layers=2, vocab_size=300, pad_token_id=0, **over))
        with pytest.raises(cabi.AdaptiveB200Error):
            cabi.Encoder.from_hf(m)
    assert torch.cuda.memory_allocated() == before


# ------------------------------------------------------------------------------------------------
# through the classifier: a seeded tiny ModernBERT opened from a directory like any hub checkpoint
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny_dir():
    from transformers import BertTokenizerFast, ModernBertConfig, ModernBertModel
    from oracle import tiny_bert
    cfg = ModernBertConfig(vocab_size=len(tiny_bert.VOCAB), hidden_size=128, num_hidden_layers=3, num_attention_heads=2,
                           intermediate_size=192, pad_token_id=0, cls_token_id=2, sep_token_id=3, bos_token_id=2,
                           eos_token_id=3, local_attention=8)
    torch.manual_seed(21)
    m = ModernBertModel(cfg).eval()
    with torch.no_grad():
        m.embeddings.tok_embeddings.weight.mul_(20.0)          # token identity survives to the CLS row
    d = tempfile.mkdtemp(prefix="tiny_modernbert_")
    m.save_pretrained(d)
    BertTokenizerFast(vocab={w: i for i, w in enumerate(tiny_bert.VOCAB)}, do_lower_case=True).save_pretrained(d)
    return d


def _texts(n, seed):
    rng = np.random.default_rng(seed)
    return [" ".join(f"w{int(i)}" for i in rng.integers(0, 195, size=int(rng.integers(3, 14)))) for _ in range(n)]


def test_classifier_on_a_modernbert_checkpoint(tiny_dir):
    import adaptive_classifier_b200 as acb
    from transformers import AutoModel, AutoTokenizer
    clf = acb.AdaptiveClassifier(tiny_dir, device="cuda")
    texts = _texts(12, 0)
    emb = torch.stack(clf._get_embeddings(texts))
    hf = AutoModel.from_pretrained(tiny_dir).eval()
    tok = AutoTokenizer.from_pretrained(tiny_dir)
    inp = tok(texts, max_length=clf.config.max_length, truncation=True, padding=True, return_tensors="pt")
    with torch.no_grad():
        ref = torch.nn.functional.normalize(hf(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"])
                                            .last_hidden_state[:, 0], dim=1)
    _check(emb, ref)

    labels = [["a", "b", "c"][i % 3] for i in range(12)]
    clf.add_examples(texts, labels)
    tests = _texts(5, 1)
    single = [clf.predict(t, k=3) for t in tests]
    batch = clf.predict_batch(tests, k=3)
    assert [[l for l, _ in p] for p in single] == [[l for l, _ in p] for p in batch]
    ids, mask, _ = clf._tokenize(tests)
    got = clf.predict_batch_ids(ids, mask, k=3)
    assert [[l for l, _ in p] for p in got] == [[l for l, _ in p] for p in batch]
    assert np.allclose([s for p in got for _, s in p], [s for p in batch for _, s in p], atol=1e-6)

    d = tempfile.mkdtemp(prefix="acb_modernbert_save_")
    clf.save(d)
    clf2 = acb.AdaptiveClassifier.load(d, device="cuda")
    a, b = clf.predict(tests[0], k=3), clf2.predict(tests[0], k=3)
    assert [l for l, _ in a] == [l for l, _ in b] and np.allclose([s for _, s in a], [s for _, s in b], atol=1e-5)
