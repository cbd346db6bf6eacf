"""CPU tests of the ModernBERT encoder path: the fp32 restatement (tests/modernbert_oracle.py) is pinned against HF
ModernBertModel (eager and sdpa), the window bound is shown to matter at the GPU tests' tolerance, and the config helper
accepts the published shapes and refuses what the CUDA path does not implement."""
import pytest
import torch

import modernbert_oracle as mo
from adaptive_classifier_b200 import _cabi

SMALL_WINDOW = dict(
    num_hidden_layers=4, norm_bias=True, attention_bias=True, mlp_bias=True, local_attention=16,
    layer_types=["sliding_attention", "full_attention", "sliding_attention", "sliding_attention"],
    rope_parameters={"sliding_attention": {"rope_type": "default", "rope_theta": 500.0},
                     "full_attention": {"rope_type": "default", "rope_theta": 20000.0}})


def _hf(m, ids, mask, impl):
    m.set_attn_implementation(impl)
    with torch.no_grad():
        hs = m(input_ids=ids, attention_mask=mask).last_hidden_state
    return torch.nn.functional.normalize(hs[:, 0], dim=1), hs


def _check(over, B, S, pads, seed):
    sd, cfg, m = mo.make_modernbert_state_dict(seed, gamma_noise=0.2, **over)
    ids = mo.synthetic_ids(B, S, vocab=cfg.vocab_size)
    mask = torch.ones_like(ids)
    for b, n in pads.items():
        mask[b, n:] = 0
    unit, hid = mo.modernbert_forward_cls(sd, ids, mask, cfg, return_hidden=True)
    valid = mask.bool()
    for impl in ("eager", "sdpa"):
        ref_unit, ref_hid = _hf(m, ids, mask, impl)
        assert (unit - ref_unit).abs().max() < 2e-6, impl
        assert (hid - ref_hid)[valid].abs().max() < 2e-6, impl


def test_oracle_matches_hf_base_dims_with_padding_beyond_the_window():
    # S = 150 > 2 * sliding_window: sliding layers really cut keys; rows 1 and 2 padded
    _check(dict(num_hidden_layers=4), 3, 150, {1: 120, 2: 9}, seed=3)


def test_oracle_matches_hf_biases_custom_layer_types_thetas_small_window():
    _check(SMALL_WINDOW, 3, 40, {1: 31, 2: 5}, seed=4)


def test_exclusive_window_is_visible_at_the_gpu_tolerance():
    """an off-by-one window (|q - k| < w instead of <= w) moves the unit CLS rows by more than 10x the 1e-3 the GPU tests
    allow, so those tests would catch it"""
    sd, cfg, _ = mo.make_modernbert_state_dict(4, gamma_noise=0.2, **SMALL_WINDOW)
    ids = mo.synthetic_ids(4, 40, vocab=cfg.vocab_size)
    inc = mo.modernbert_forward_cls(sd, ids, None, cfg)
    exc = mo.modernbert_forward_cls(sd, ids, None, cfg, inclusive_window=False)
    assert (inc - exc).norm(dim=1).max() > 1e-2


def test_layer_windows_follow_the_config():
    from transformers import ModernBertConfig
    c = ModernBertConfig()
    wins, thetas = mo.layer_windows_thetas(c)
    assert wins[:4] == [0, 64, 64, 0] and thetas[:4] == [160000.0, 10000.0, 10000.0, 160000.0]
    d = _cabi.modernbert_dims(c)
    assert d["windows"] == wins and d["thetas"] == thetas


def test_config_helper_accepts_base_and_large():
    from transformers import ModernBertConfig
    base = _cabi.modernbert_dims(ModernBertConfig())
    assert (base["layers"], base["hidden"], base["heads"], base["intermediate"], base["vocab"]) == (22, 768, 12, 1152, 50368)
    assert base["norm_eps"] == 1e-5
    large = _cabi.modernbert_dims(ModernBertConfig(num_hidden_layers=28, hidden_size=1024, num_attention_heads=16,
                                                   intermediate_size=2624))
    assert (large["layers"], large["hidden"], large["heads"], large["intermediate"]) == (28, 1024, 16, 2624)
    assert len(large["windows"]) == 28


@pytest.mark.parametrize("over, what", [
    (dict(hidden_activation="gelu_pytorch_tanh"), "hidden_activation"),
    (dict(rope_parameters={"sliding_attention": {"rope_type": "linear", "rope_theta": 1e4, "factor": 2.0},
                           "full_attention": {"rope_type": "default", "rope_theta": 1.6e5}}), "rope"),
    (dict(rope_parameters={"sliding_attention": {"rope_type": "default", "rope_theta": 1e4},
                           "full_attention": {"rope_type": "default", "rope_theta": 1.6e5, "factor": 2.0}}), "rope"),
    (dict(hidden_size=768, num_attention_heads=6), "head_dim"),
    (dict(hidden_size=704, num_attention_heads=11), "hidden_size"),
    (dict(hidden_size=1152, num_attention_heads=18), "hidden_size"),
    (dict(intermediate_size=1000), "intermediate_size"),
])
def test_config_helper_rejects_what_is_not_implemented(over, what):
    from transformers import ModernBertConfig
    c = ModernBertConfig(**{k: v for k, v in over.items() if k != "rope_parameters"})
    if "rope_parameters" in over:
        c.rope_parameters = over["rope_parameters"]
    with pytest.raises(_cabi.AdaptiveB200Error, match=what):
        _cabi.modernbert_dims(c)


def test_geglu_chunk_order_restated():
    """the Wi packing of ac_encoder_create_modernbert (packed row 32 q + j = input row 16 q + j for j < 16, gate row
    I + 16 q + j - 16 otherwise) followed by the epilogue's pairing (column j of a 32-column chunk with column j + 16)
    equals input, gate = chunk(2)"""
    I, H, T = 128, 64, 5
    W = torch.randn(2 * I, H, dtype=torch.float64)
    x = torch.randn(T, H, dtype=torch.float64)
    p = torch.arange(2 * I)
    q, j = p // 32, p % 32
    src = torch.where(j < 16, 16 * q + j, I + 16 * q + j - 16)
    acc = x @ W[src].t()                                   # the GEMM over the packed rows
    a = acc.view(T, 2 * I // 32, 32)
    out = (a[..., :16] * a[..., 16:]).reshape(T, I)        # output column 16 q + j of chunk q
    inp, gate = (x @ W.t()).chunk(2, dim=-1)
    assert torch.equal(out, inp * gate)
