"""fp64 CPU reference of the encoder's attention (ac_attention: attention_kernel / attention_long_kernel in csrc/encoder.cu) and
the seeded inputs its tests run on.  Test infrastructure only.

The reference takes the same fp16 tensors the kernels receive:
    scores = q . k / 8 over the visible keys (key k < S, mask[b, k] != 0 and, when windowed, |q - k| <= window);
    P = exp(scores - max) (optionally rounded to fp16, as the kernels round P before the P V product);
    ctx = P V / sum(unrounded P); a row with no visible key gives zeros, as the kernels document.

The inputs make attention sharp, so that one key matters to one query row:
  - Q and K have a score std of about 10 after the 1/8 scale (spreads of +-20-40, which also exercises the max subtraction);
  - planted rows put their single best key (logit +40, the others ~N(0, 5^2)) at key 0, keys 127 / 128 / 255 / 256 / 383 / 384,
    the last valid key and keys exactly `window` away; decoy rows aim the same way at a key just OUTSIDE the window;
  - planted two-key rows split P between two keys 1.5 logits apart with V = +1 / -1, where a scale error moves P the most;
  - every position the kernels must ignore holds BIG = 3e4 (finite: 0 * BIG = 0): the K rows and V^T columns of masked keys,
    V^T columns S .. S_pad - 1 and the Q/K rows past B*S that the 128-row tiles read.  A mask applied wrongly is an O(1e4)
    error, not a rounding-level one.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch

BIG = 3.0e4
Q_STD = 10.0 ** 0.5          # q . k / 8 over 64 dims of N(0, 10) products: std 64^0.5 * 10 / 8 = 10
PLANT_LOGIT = 40.0
PAIR_GAP = 1.5               # d/dlambda sigmoid(lambda g) = g s (1 - s) peaks near g = 1.5
MASK_KINDS = ("none", "suffix", "left", "holes", "cls_only")

# Tolerance per element of ctx, in units of 2^-11 max|v| (max|v| = 1 by construction).  With P rounded to fp16 in the reference
# as in the kernels, what is left is the fp16 rounding of ctx (<= 2^-12 for |ctx| < 1), an occasional fp16 rounding of one P
# that falls the other way because ex2.approx (~2^-22 relative) and the fp32 scores differ from fp64 (one fp16 ulp of that P,
# <= 2^-11 |v| for P < 1/2), and fp32 accumulation (~1e-7): about 1.5 units at worst.  Measured on an NVIDIA B200 (1000 W)
# over the whole grid of the GPU test: 1.11 units (5.4e-4) at most.
TOL_UNITS = 2.0


def roundup8(S: int) -> int:
    return (S + 7) // 8 * 8


def make_mask(kind: str, B: int, S: int, g: torch.Generator) -> Optional[torch.Tensor]:
    """int32 [B, S] (1 keep / 0 pad) or None"""
    if kind == "none":
        return None
    m = torch.ones(B, S, dtype=torch.int32)
    for b in range(B):
        if kind == "suffix":                       # sequence b keeps its first n keys
            m[b, max(1, S - (b + 1) * S // (B + 2) - b):] = 0
        elif kind == "left":                       # sequence b loses its first p keys
            m[b, :min(S - 1, (b + 1) * S // (B + 2) + b)] = 0
        elif kind in ("holes", "cls_only"):        # a quarter of the keys missing, key 0 kept
            m[b] = (torch.rand(S, generator=g) >= 0.25).to(torch.int32)
            m[b, 0] = 1
        else:
            raise ValueError(kind)
    if kind == "cls_only":
        m[0] = 0
        m[0, 0] = 1                                # only the CLS key is valid
        if B > 1:
            m[1] = 0                               # no key at all: every row of this sequence is zero
    return m


def visibility(mask: Optional[torch.Tensor], B: int, S: int, window: int) -> torch.Tensor:
    """bool [B, S (query), S (key)]; window 0 = global"""
    valid = torch.ones(B, S, dtype=torch.bool) if mask is None else mask.to(torch.bool)
    vis = valid[:, None, :].expand(B, S, S).clone()
    if window > 0:
        pos = torch.arange(S)
        vis &= ((pos[:, None] - pos[None, :]).abs() <= window)[None]
    return vis


def _plants(S: int, window: int) -> Tuple[List[Tuple[int, int]], List[Tuple[int, int]], List[Tuple[int, int, int]]]:
    """(query, best key) targets, (query, decoy key outside the window) and (query, key +1, key -1) two-key rows"""
    best = [(0, 0), (S - 1, 0), (S // 2, 0), (128, 0), (129, 0), (200, 0), (300, 0), (511, 0)]
    for kk in (31, 32, 63, 64, 127, 128, 255, 256, 383, 384, 511):
        best += [(kk, kk), (kk + 3, kk), (kk - 5, kk), (S - 2, kk)]
    best += [(S // 3, S - 1), (S - 1, S - 1)]
    decoy = []
    if window > 0:
        for q in (0, 1, S // 2, S - 1, 127, 128, 130, 255, 256, 300):
            best += [(q, q + window), (q + 1, q + 1 - window)]
            decoy += [(q + 2, q + 2 + window + 1), (q + 3, q + 3 - window - 1)]
    pairs = [(S // 4, S // 4, S // 4 + 1), (S - 1, S - 1, S - 2), (130, 130, 2), (5, 4, 5)]
    return best, decoy, pairs


def make_inputs(B: int, S: int, heads: int, mask_kind: str, window: int = 0, seed: int = 0):
    """-> dict(qk fp16 [B*S + 128, 2H], vT fp16 [B*H, S_pad], mask int32 [B, S] or None, B, S, heads, window)"""
    g = torch.Generator().manual_seed(seed * 1000003 + B * 7919 + S * 31 + heads * 7 + window)
    H, S_pad = 64 * heads, roundup8(S)
    mask = make_mask(mask_kind, B, S, g)
    valid = torch.ones(B, S, dtype=torch.bool) if mask is None else mask.to(torch.bool)
    vis = visibility(mask, B, S, window)
    q = torch.randn(B, S, heads, 64, generator=g, dtype=torch.float64) * Q_STD
    k = (torch.randn(B, S, heads, 64, generator=g, dtype=torch.float64) * Q_STD).half().double()
    v = torch.rand(B, S, heads, 64, generator=g, dtype=torch.float64) * 2 - 1
    best, decoy, pairs = _plants(S, window)
    ok = lambda i: 0 <= i < S
    for b in range(B):
        used = set()                                                       # one plant per query row, first one wins
        for qi, ki in best + decoy:
            if ok(qi) and ok(ki) and qi not in used and valid[b, ki] and (vis[b, qi, ki] or (qi, ki) in decoy):
                kv = k[b, ki]                                              # [heads, 64]
                q[b, qi] = kv * (8 * PLANT_LOGIT / (kv * kv).sum(-1, keepdim=True))
                used.add(qi)
        for qi, k1, k2 in pairs:
            if ok(qi) and ok(k1) and ok(k2) and k1 != k2 and qi not in used and vis[b, qi, k1] and vis[b, qi, k2]:
                a, c = k[b, k1], k[b, k2]
                g11, g12, g22 = (a * a).sum(-1), (a * c).sum(-1), (c * c).sum(-1)
                r1, r2 = 8 * PLANT_LOGIT, 8 * (PLANT_LOGIT - PAIR_GAP)
                det = g11 * g22 - g12 * g12
                al, be = (r1 * g22 - r2 * g12) / det, (r2 * g11 - r1 * g12) / det
                q[b, qi] = al[:, None] * a + be[:, None] * c
                v[b, k1], v[b, k2] = 1.0, -1.0
                used.add(qi)
    qk = torch.full((B * S + 128, 2 * H), BIG, dtype=torch.float16)
    qk[:B * S, :H] = q.reshape(B * S, H).half()
    kk = k.clone()
    kk[~valid] = BIG
    qk[:B * S, H:] = kk.reshape(B * S, H).half()
    vt = torch.full((B, heads, 64, S_pad), BIG, dtype=torch.float64)
    vv = v.clone()
    vv[~valid] = BIG
    vt[..., :S] = vv.permute(0, 2, 3, 1)
    return dict(qk=qk, vT=vt.reshape(B * H, S_pad).half(), mask=mask, B=B, S=S, heads=heads, window=window)


def attention_ref(qk: torch.Tensor, vT: torch.Tensor, mask: Optional[torch.Tensor], B: int, S: int, heads: int, window: int,
                  *, round_p: bool = True, scale: float = 0.125, vis: Optional[torch.Tensor] = None):
    """-> (ctx float64 [B*S, H], has_key bool [B*S]).  `vis` [B, S, S] overrides the visibility (tests of the inputs)."""
    H = 64 * heads
    q = qk[:B * S, :H].double().view(B, S, heads, 64).transpose(1, 2)
    k = qk[:B * S, H:].double().view(B, S, heads, 64).transpose(1, 2)
    v = vT.double().view(B, heads, 64, -1)[..., :S].transpose(-1, -2)
    if vis is None:
        vis = visibility(mask, B, S, window)
    s = (q @ k.transpose(-1, -2)) * scale
    s = s.masked_fill(~vis[:, None], -math.inf)
    has = vis.any(-1)[:, None, :, None]
    mx = torch.where(has, s.amax(-1, keepdim=True), torch.zeros(()))
    e = torch.exp(s - mx)
    den = e.sum(-1, keepdim=True)
    p = e.half().double() if round_p else e
    ctx = torch.where(has, (p @ v) / torch.where(den > 0, den, torch.ones(())), torch.zeros(()))
    return ctx.transpose(1, 2).reshape(B * S, H), vis.any(-1).reshape(B * S)


def tolerance(inp) -> float:
    """per-element bound on |ctx - reference| (see TOL_UNITS)"""
    B, S, heads = inp["B"], inp["S"], inp["heads"]
    v = inp["vT"].double().view(B, heads, 64, -1)[..., :S]
    valid = torch.ones(B, S, dtype=torch.bool) if inp["mask"] is None else inp["mask"].to(torch.bool)
    vmax = v.abs().amax(dim=(1, 2))[valid].max().item() if bool(valid.any()) else 1.0
    return TOL_UNITS * 2.0 ** -11 * vmax


# ---- the grid the GPU test runs: every S edge with every mask kind (global), and windows on both sides of 128 ----
S_EDGES = (1, 2, 3, 7, 8, 9, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 383, 385, 511, 512)
B_CYCLE = (1, 3, 7)
HEADS_CYCLE = (1, 2, 12, 16)
WIN_S = (100, 128, 129, 300, 512)


def window_list(S: int) -> List[int]:
    return sorted({w for w in (1, 2, 8, 31, 32, 63, 64, 127, 128, S - 2, S - 1, S) if w > 0})


def grid() -> List[Tuple[int, int, int, str, int]]:
    """(B, S, heads, mask kind, window) cases"""
    cases = []
    for i, S in enumerate(S_EDGES):
        for j, kind in enumerate(MASK_KINDS):
            cases.append((B_CYCLE[(i + j) % 3], S, HEADS_CYCLE[(i + 2 * j) % 4], kind, 0))
    for i, S in enumerate(WIN_S):
        for j, w in enumerate(window_list(S)):
            cases.append((B_CYCLE[(i + j) % 3], S, HEADS_CYCLE[(i + j) % 4], MASK_KINDS[(i + j) % len(MASK_KINDS)], w))
    return cases
