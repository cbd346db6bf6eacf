"""CPU tests of tests/attention_reference.py: the reference is plain softmax attention, and the GPU test's inputs are sharp
enough that each simulated attention bug below moves the reference's output by at least 10x the GPU tolerance on a row the
GPU test asserts.  An edit that makes the inputs blind to one of these bugs fails here, before any GPU time is spent."""
import math

import pytest
import torch

import attention_reference as ar


def _case(B, S, heads, kind, window):
    assert (B, S, heads, kind, window) in ar.grid(), "sensitivity is checked on cases the GPU test runs"
    return ar.make_inputs(B, S, heads, kind, window)


def test_reference_is_softmax_attention():
    inp = ar.make_inputs(3, 40, 2, "holes", 0)
    ctx, has = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], 3, 40, 2, 0, round_p=False)
    q = inp["qk"][:120, :128].double().view(3, 40, 2, 64).transpose(1, 2)
    k = inp["qk"][:120, 128:].double().view(3, 40, 2, 64).transpose(1, 2)
    v = inp["vT"].double().view(3, 2, 64, 40).transpose(-1, -2)
    add = (1.0 - inp["mask"].double())[:, None, None, :] * -1e300
    want = (torch.softmax(q @ k.transpose(-1, -2) / 8 + add, -1) @ v).transpose(1, 2).reshape(120, 128)
    assert bool(has.all()) and (ctx - want).abs().max().item() < 1e-12
    # rounding P to fp16 stays inside the tolerance
    ctx16, _ = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], 3, 40, 2, 0)
    assert (ctx16 - ctx).abs().max().item() < ar.tolerance(inp) / 2


def test_rows_without_a_visible_key_are_zero_and_ignored_positions_hold_big():
    inp = ar.make_inputs(3, 65, 2, "cls_only", 8)
    ctx, has = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], 3, 65, 2, 8)
    has = has.view(3, 65)
    assert bool(has[0, :9].all()) and not bool(has[0, 9:].any()) and not bool(has[1].any())
    assert bool((ctx.view(3, 65, -1)[~has] == 0).all())
    assert bool((inp["qk"][3 * 65:] == ar.BIG).all())                              # rows past B*S
    assert bool((inp["vT"][:, 65:] == ar.BIG).all())                               # V^T columns S .. S_pad - 1
    assert bool((inp["qk"][65:130, 128:] == ar.BIG).all())                         # K rows of sequence 1 (all masked)


def _moved(inp, **mut):
    B, S, h, w = inp["B"], inp["S"], inp["heads"], inp["window"]
    ref, has = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], B, S, h, w)
    bad, _ = ar.attention_ref(inp["qk"], inp["vT"], inp["mask"], B, S, h, w, **mut)
    return (bad - ref)[has].abs().max().item() / ar.tolerance(inp)


def _vis(inp):
    return ar.visibility(inp["mask"], inp["B"], inp["S"], inp["window"])


def _window_lt(inp):                          # |q - k| < w instead of <= w
    S = inp["S"]
    pos = torch.arange(S)
    valid = torch.ones(inp["B"], S, dtype=torch.bool) if inp["mask"] is None else inp["mask"].bool()
    return valid[:, None, :] & ((pos[:, None] - pos[None, :]).abs() < inp["window"])[None]


def _mutations():
    out = []

    def key0_lost_for_rows_ge_128(inp):
        v = _vis(inp); v[:, 128:, 0] = False; return dict(vis=v)

    def last_key_of_each_block_dropped(inp):
        v = _vis(inp); v[..., 127::128] = False; return dict(vis=v)

    def query_block_1_ignores_the_mask(inp):
        v = _vis(inp); v[:, 128:256] = ar.visibility(None, inp["B"], inp["S"], inp["window"])[:, 128:256]; return dict(vis=v)

    def window_plus_one(inp):
        return dict(vis=ar.visibility(inp["mask"], inp["B"], inp["S"], inp["window"] + 1))

    def window_minus_one(inp):
        return dict(vis=_window_lt(inp))

    def scale_times_1_05(inp):
        return dict(scale=0.125 * 1.05)

    def mask_word_shifted_by_32(inp):
        m, n = inp["mask"].clone(), min(64, inp["S"]) - 32
        m[:, 32:32 + n] = inp["mask"][:, 0:n]
        return dict(vis=ar.visibility(m, inp["B"], inp["S"], inp["window"]))

    for fn, cases in ((key0_lost_for_rows_ge_128, [(7, 129, 12, "none", 0), (3, 385, 16, "none", 0)]),
                      (last_key_of_each_block_dropped, [(7, 257, 2, "none", 0), (3, 128, 2, "none", 0)]),
                      (query_block_1_ignores_the_mask, [(1, 257, 16, "suffix", 0), (3, 385, 2, "holes", 0)]),
                      (window_plus_one, [(7, 100, 12, "left", 8), (3, 300, 16, "left", 32), (7, 512, 16, "suffix", 127)]),
                      (window_minus_one, [(7, 100, 12, "left", 8), (3, 300, 16, "left", 32), (7, 512, 16, "suffix", 127)]),
                      (scale_times_1_05, [(3, 64, 1, "holes", 0), (1, 512, 2, "none", 0), (7, 300, 2, "none", 8)]),
                      (mask_word_shifted_by_32, [(1, 63, 16, "holes", 0), (7, 257, 16, "holes", 0), (7, 512, 1, "holes", 32)])):
        for c in cases:
            out.append(pytest.param(fn, c, id=f"{fn.__name__}-B{c[0]}-S{c[1]}-h{c[2]}-{c[3]}-w{c[4]}"))
    return out


@pytest.mark.parametrize("mutate,case", _mutations())
def test_each_simulated_bug_moves_an_asserted_row_by_10x_the_tolerance(mutate, case):
    inp = _case(*case)
    moved = _moved(inp, **mutate(inp))
    assert math.isfinite(moved) and moved >= 10.0, moved
