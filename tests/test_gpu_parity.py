"""GPU parity tests proper: every call goes through the C ABI (ctypes) and is compared with the CPU oracle
on the same seeded inputs.  Bit-exact for indices and lane-ordered distances; stated tolerances for fp32 math."""
import numpy as np
import pytest
import torch

from oracle import encoder_oracle as eo
from oracle import head_oracle as ho
from oracle import knn_oracle as ko

pytestmark = pytest.mark.gpu


def _unit(x):
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def _synthetic_index(N, D, C, seed=0):
    """SURVEY.md section 8(d): class centres (always Generator(0)) + 0.5-norm noise (Generator(seed+100)),
    row j belongs to class j mod C; seed 0 = index rows, seed 1 = queries around the same centres."""
    centres = torch.nn.functional.normalize(torch.randn(C, D, generator=torch.Generator().manual_seed(0)), dim=1)
    g = torch.Generator().manual_seed(seed + 100)
    noise = torch.randn(N, D, generator=g) * (0.5 / D ** 0.5)
    rows = torch.nn.functional.normalize(centres[torch.arange(N) % C] + noise, dim=1)
    return rows.contiguous(), centres


def _tf32(t):
    return eo.round_tf32(t.float().cpu()).to(t.device)


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K,epi", [(256, 256, 64, 0), (1000, 768, 768, 2), (4096, 3072, 768, 1), (300, 80, 96, 0),
                                       (128, 2304, 768, 0)])
def test_linear_tc_matches_fp64(cabi, M, N, K, epi):
    g = torch.Generator().manual_seed(M + N + K)
    X = _tf32(torch.randn(M, K, generator=g))
    W = _tf32(torch.randn(N, K, generator=g) * 0.05)
    b = torch.randn(N, generator=g)
    R = torch.randn(M, N, generator=g)
    ref = X.double() @ W.double().t() + b.double()
    if epi == 1:
        ref = 0.5 * ref * (1 + torch.erf(ref / 2 ** 0.5))
    if epi == 2:
        ref = ref + R.double()
    Y = cabi.linear_tc(X.cuda(), W.cuda(), b.cuda(), R.cuda() if epi == 2 else None, epi=epi).cpu()
    err = (Y.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    # operands are exact tf32 values, products exact in fp32, only the fp32 accumulation order differs
    assert err <= 2e-5 * max(scale, 1.0), (err, scale)


@pytest.mark.parametrize("M,N,K,epi,out_half", [(256, 256, 64, 0, True), (1000, 768, 768, 2, False), (4096, 3072, 768, 1, True),
                                                  (300, 80, 128, 0, False), (128, 2304, 768, 0, True), (77, 768, 3072, 2, False)])
def test_linear_f16_matches_fp64(cabi, M, N, K, epi, out_half):
    """the encoder's GEMM: fp16 operands (exact products), fp32 accumulation in TMEM, fused epilogues"""
    g = torch.Generator().manual_seed(M + N + K + 1)
    X = torch.randn(M, K, generator=g).half()
    W = (torch.randn(N, K, generator=g) * 0.05).half()
    b = torch.randn(N, generator=g)
    R = torch.randn(M, N, generator=g)
    ref = X.double() @ W.double().t() + b.double()
    if epi == 1:
        ref = 0.5 * ref * (1 + torch.erf(ref / 2 ** 0.5))
    if epi == 2:
        ref = ref + R.double()
    Y = cabi.linear_tc(X.cuda(), W.cuda(), b.cuda(), R.cuda() if epi == 2 else None, epi=epi, out_half=out_half).cpu()
    assert Y.dtype == (torch.float16 if out_half else torch.float32)
    err = (Y.double() - ref).abs().max().item()
    scale = max(ref.abs().max().item(), 1.0)
    # fp32 accumulation order + the 1.5e-7 erf approximation; fp16 output adds one rounding (2^-11 relative)
    assert err <= (1e-3 if out_half else 3e-5) * scale, (err, scale)


# ------------------------------------------------------------------------------------------------ kNN exact
@pytest.mark.parametrize("B,N,D,k", [(1, 5000, 768, 5), (3, 5000, 768, 64), (8, 1000, 768, 1000), (20, 3000, 1024, 7),
                                     (5, 257, 10, 3), (2, 3, 768, 5), (1, 20000, 768, 1000)])
def test_knn_exact_bit_identical(cabi, B, N, D, k):
    rng = np.random.default_rng(B * 1000 + N)
    Q = _unit(rng.standard_normal((B, D)).astype(np.float32))
    P = _unit(rng.standard_normal((N, D)).astype(np.float32))
    P[N // 2] = P[N // 3]            # an exact duplicate row: tie must go to the lower id
    d_ref, i_ref = ko.knn_l2(Q, P, k, row_offset=11)
    d, i = cabi.knn_l2_topk(torch.from_numpy(Q).cuda(), torch.from_numpy(P).cuda(), k, row_offset=11,
                            algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    assert np.array_equal(i.cpu().numpy(), i_ref)
    assert np.array_equal(d.cpu().numpy(), d_ref)     # same lane order -> same bits (inf == inf for padding)


def test_knn_tensor_path_identical_to_oracle(cabi):
    B, N, D, C, k = 64, 20000, 768, 20, 5
    P, centres = _synthetic_index(N, D, C, seed=0)
    Qr, _ = _synthetic_index(B, D, C, seed=1)
    d_ref, i_ref = ko.knn_l2(Qr.numpy(), P.numpy(), k)
    d, i = cabi.knn_l2_topk(Qr.cuda(), P.cuda(), k, algo=cabi.AC_KNN_TENSOR)
    torch.cuda.synchronize()
    assert np.array_equal(i.cpu().numpy(), i_ref)
    assert np.array_equal(d.cpu().numpy(), d_ref)


@pytest.mark.parametrize("B,N,C,k", [(256, 100_000, 20, 5), (512, 300_000, 1000, 5), (130, 70_001, 50, 16)])
def test_knn_tensor_equals_exact_scan_large(cabi, B, N, C, k):
    """Full-size property: tensor path == exact scan on the GPU, bit for bit (the exact scan is pinned
    against the oracle above)."""
    D = 768
    P, _ = _synthetic_index(N, D, C, seed=0)
    Q, _ = _synthetic_index(B, D, C, seed=1)
    Pg, Qg = P.cuda(), Q.cuda()
    d1, i1 = cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_TENSOR)
    d0, i0 = cabi.knn_l2_topk(Qg[:32], Pg, k, algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    assert torch.equal(i1[:32], i0)
    assert torch.equal(d1[:32], d0)
    # top-1 label of a query = its own class (rows j belong to class j mod C)
    assert torch.equal(i1[:, 0].cpu() % C, torch.arange(B) % C)
    # ascending order
    assert bool((d1[:, 1:] >= d1[:, :-1]).all())


@pytest.mark.parametrize("B,N,C,k", [(512, 200_000, 1000, 5), (96, 50_000, 20, 16)])
def test_knn_tensor_fp16_shadow_equals_exact_scan(cabi, B, N, C, k):
    """coarse pass over the fp16 shadow (kind::f16, 2.N.D bytes) + exact fp32 re-rank + certification == exact scan"""
    D = 768
    P, _ = _synthetic_index(N, D, C, seed=0)
    Q, _ = _synthetic_index(B, D, C, seed=1)
    Pg, Qg = P.cuda(), Q.cuda()
    Ph = cabi.knn_make_shadow(Pg)
    assert Ph.dtype == torch.float16 and torch.equal(Ph, Pg.half())
    d1, i1 = cabi.knn_l2_topk(Qg, Pg, k, p_half=Ph, algo=cabi.AC_KNN_TENSOR)
    d2, i2 = cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_TENSOR)           # tf32 coarse pass on the fp32 rows
    d0, i0 = cabi.knn_l2_topk(Qg[:48], Pg, k, algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    assert torch.equal(i1, i2) and torch.equal(d1, d2)
    assert torch.equal(i1[:48], i0) and torch.equal(d1[:48], d0)
    assert torch.equal(i1[:, 0].cpu() % C, torch.arange(B) % C)


@pytest.mark.parametrize("B,N,D,C,k", [(64, 30_000, 768, 20, 64), (512, 120_000, 768, 1000, 1000), (130, 50_000, 1024, 50, 200),
                                       (700, 60_000, 768, 100, 100)])
def test_knn_tensor_large_k_equals_exact_scan(cabi, B, N, D, C, k):
    """k = num_classes (predict() semantics, classifier.py:424-425) stays on the tensor path: pass 1 bounds the k-th distance,
    pass 2 collects the provable superset {coarse <= tau + 2 eps}, exact re-rank + (d, id) selection.  B = 700 runs as two
    query blocks.  Bit-identical to the exact scan (sample of queries) and to the oracle (4 queries)."""
    P, _ = _synthetic_index(N, D, C, seed=0)
    Q, _ = _synthetic_index(B, D, C, seed=1)
    Pg, Qg = P.cuda(), Q.cuda()
    Ph = cabi.knn_make_shadow(Pg)
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    d1, i1 = cabi.knn_l2_topk(Qg, Pg, k, p_half=Ph, algo=cabi.AC_KNN_TENSOR, stats=stats)
    sel = torch.arange(0, B, max(1, B // 24))[:24]
    d0, i0 = cabi.knn_l2_topk(Qg[sel.cuda()].contiguous(), Pg, k, algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    st = stats.cpu().tolist()
    assert st[1] == 0 and st[0] == B and k <= st[2] <= 4096, st           # every query took pass 2, nothing overflowed
    assert torch.equal(i1[sel.cuda()], i0) and torch.equal(d1[sel.cuda()], d0)
    assert bool((d1[:, 1:] >= d1[:, :-1]).all())
    d_ref, i_ref = ko.knn_l2(Q[:4].numpy(), P.numpy(), k)
    assert np.array_equal(i1[:4].cpu().numpy(), i_ref) and np.array_equal(d1[:4].cpu().numpy(), d_ref)


def test_knn_tensor_near_duplicate_rows_take_the_second_pass_not_a_full_scan(cabi):
    """Stress input of VERDICT r1 #14: every query has MANY rows closer to each other than the coarse error bound
    (gaps < eps ~ 2e-3), so pass-1 certification fails for all of them.  They are resolved by the second tensor pass
    (device-conditional, no host sync) -- bit-identical to the exact scan, ties by lower row id, and stats say so."""
    B, N, D, k = 256, 80_000, 768, 5
    g = torch.Generator().manual_seed(3)
    base = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    P = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
    for b in range(B):                      # 48 near-copies of every query's neighbour, 1e-4 apart, scattered over the index:
        rows = (torch.arange(48) * 1601 + b * 311) % N          # more than the 32 re-ranked candidates -> T - eps < d_k
        P[rows] = torch.nn.functional.normalize(base[b][None] + 1e-4 * torch.randn(48, D, generator=g), dim=1)
    P[5] = P[40_005]                        # an exact duplicate: tie -> lower id
    Q = torch.nn.functional.normalize(base + 1e-3 * torch.randn(B, D, generator=g), dim=1)
    Pg, Qg = P.cuda().contiguous(), Q.cuda().contiguous()
    Ph = cabi.knn_make_shadow(Pg)
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    d1, i1 = cabi.knn_l2_topk(Qg, Pg, k, p_half=Ph, algo=cabi.AC_KNN_TENSOR, stats=stats)
    d0, i0 = cabi.knn_l2_topk(Qg[:64].contiguous(), Pg, k, algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    st = stats.cpu().tolist()
    assert st[0] >= B // 2 and st[1] == 0, st          # most queries could not be certified; none overflowed
    assert torch.equal(i1[:64], i0) and torch.equal(d1[:64], d0)
    # synchronous mode (no stats pointer) gives the same answer
    d2, i2 = cabi.knn_l2_topk(Qg, Pg, k, p_half=Ph, algo=cabi.AC_KNN_TENSOR)
    assert torch.equal(i2, i1) and torch.equal(d2, d1)


def test_knn_tensor_overflow_is_reported_and_rescued(cabi):
    """thousands of identical rows inside the 2-eps band overflow the candidate buffer: with a stats pointer the overflow is
    reported (stats[1]); without one the call recomputes those queries by the exact scan"""
    B, N, D, k = 32, 20_000, 768, 5
    g = torch.Generator().manual_seed(8)
    P = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
    P[1000:1600] = P[999]                                          # 600 identical rows > cap (256 for k <= 16)
    Q = torch.nn.functional.normalize(P[999][None] + 0.01 * torch.randn(B, D, generator=g), dim=1)
    Pg, Qg = P.cuda().contiguous(), Q.cuda().contiguous()
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_TENSOR, stats=stats)
    assert stats.cpu().tolist()[1] == B
    d1, i1 = cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_TENSOR)          # synchronous mode rescues
    d0, i0 = cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_EXACT)
    assert torch.equal(i1, i0) and torch.equal(d1, d0)
    assert i1[0].tolist() == [999, 1000, 1001, 1002, 1003]                  # ties -> lower row id


@pytest.mark.parametrize("N,D,B", [(1_000_000, 768, 512), (500_000, 1024, 128)])
def test_knn_tensor_at_the_benched_sizes_equals_oracle(cabi, N, D, B):
    """BASELINE configs[2] (1 M x 768, 512 queries) and configs[4] (500 k x 1024, 128 queries): the sizes bench.py runs, against
    the ORACLE on a 32-query sample (bit-exact ids and distances) and the exact scan on the same sample"""
    from adaptive_classifier_b200 import workload as wl
    C, k = (1000, 5) if D == 768 else (50, 5)
    P = wl.synthetic_rows(0, N, D, C, seed=0, device="cuda")
    Q = wl.synthetic_queries_embeddings(B, D, C, device="cuda")
    Ph = cabi.knn_make_shadow(P)
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    d1, i1 = cabi.knn_l2_topk(Q, P, k, p_sqnorm=cabi.row_sqnorm(P), p_half=Ph, algo=cabi.AC_KNN_TENSOR, stats=stats)
    sel = torch.arange(0, B, B // 32)[:32].cuda()
    d0, i0 = cabi.knn_l2_topk(Q[sel].contiguous(), P, k, algo=cabi.AC_KNN_EXACT)
    torch.cuda.synchronize()
    assert stats.cpu().tolist()[1] == 0
    assert torch.equal(i1[sel], i0) and torch.equal(d1[sel], d0)
    d_ref, i_ref = ko.knn_l2(Q[sel].cpu().numpy(), P.cpu().numpy(), k)
    assert np.array_equal(i1[sel].cpu().numpy(), i_ref) and np.array_equal(d1[sel].cpu().numpy(), d_ref)


def test_golden_router_prototypes_through_the_cuda_kernels(cabi):
    """tests/golden/golden_router.npz: the two REAL prototypes of the reference's bundled router (d = 0.001965 apart: the
    near-tie stress input of SURVEY 8(c)) searched by the reference-side index object -> same (d, id) bits from both CUDA paths"""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_router.npz"))
    P, Q = torch.from_numpy(g["P"]).cuda(), torch.from_numpy(g["Q"]).cuda()
    d, i = cabi.knn_l2_topk(Q, P, 2, algo=cabi.AC_KNN_EXACT)
    assert np.array_equal(i.cpu().numpy(), g["i"]) and np.array_equal(d.cpu().numpy(), g["d"])
    # the tensor path on the same rows embedded in a larger index (the two prototypes stay the nearest rows)
    filler = torch.nn.functional.normalize(torch.randn(8190, P.shape[1], generator=torch.Generator().manual_seed(1)), dim=1).cuda() * 3.0
    big = torch.cat([P, filler]).contiguous()
    Q32 = Q.repeat(3, 1)[:32].contiguous()
    dt, it = cabi.knn_l2_topk(Q32, big, 2, algo=cabi.AC_KNN_TENSOR)
    assert np.array_equal(it.cpu().numpy()[:12], g["i"]) and np.array_equal(dt.cpu().numpy()[:12], g["d"])


def test_golden_head_through_the_cuda_kernels(cabi):
    """tests/golden/golden_head.npz: the reference's AdaptiveHead logits and EWC loss values on seeded inputs"""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_head.npz"))
    names = {"W0": "model.0.weight", "b0": "model.0.bias", "W1": "model.3.weight", "b1": "model.3.bias",
             "W2": "model.6.weight", "b2": "model.6.bias"}
    pg = {k: torch.from_numpy(g[v]).cuda().contiguous() for k, v in names.items()}
    X = torch.from_numpy(g["X"]).cuda()
    logits = cabi.head_forward(X, pg, cabi.AC_ACT_LOGITS).cpu().numpy()
    assert np.abs(logits - g["logits"]).max() < 1e-5
    fisher = {k: torch.from_numpy(g["fisher_" + v]).cuda().contiguous() for k, v in names.items()}
    moved = {k: (v + 0.1).contiguous() for k, v in pg.items()}
    assert float(cabi.ewc_penalty(pg, fisher, pg, 100.0, None)) == 0.0 == float(g["ewc_loss0"])
    l1 = float(cabi.ewc_penalty(moved, fisher, pg, 100.0, None))
    assert abs(l1 - float(g["ewc_loss1"])) <= 1e-4 * float(g["ewc_loss1"])
    l32 = float(cabi.ewc_penalty(moved, fisher, pg, 100.0, 32))
    assert abs(l32 - float(g["ewc_loss1_b32"])) <= 1e-4 * float(g["ewc_loss1_b32"])


def test_proto_scores_and_merge(cabi):
    rng = np.random.default_rng(3)
    d = np.sort(rng.uniform(0, 4, size=(7, 9)).astype(np.float32), axis=1)
    idx = rng.integers(0, 100, size=(7, 9)).astype(np.int64)
    idx[2, 6:] = -1
    s_ref = ko.proto_scores(d, idx)
    s = cabi.proto_scores(torch.from_numpy(d).cuda(), torch.from_numpy(idx).cuda()).cpu().numpy()
    assert np.abs(s - s_ref).max() < 1e-6
    G, B, k = 4, 5, 6
    dd = np.sort(rng.uniform(0, 4, size=(G, B, k)).astype(np.float32), axis=2)
    ii = rng.permutation(G * B * k).reshape(G, B, k).astype(np.int64)
    dd[1, :, :] = dd[0, :, :]        # ties across shards -> lower id wins
    ii[3, 0, 3:] = -1
    od_ref, oi_ref = ko.topk_merge(dd, ii)
    od, oi = cabi.topk_merge(torch.from_numpy(dd).cuda(), torch.from_numpy(ii).cuda())
    assert np.array_equal(oi.cpu().numpy(), oi_ref) and np.array_equal(od.cpu().numpy(), od_ref)


def test_sharded_search_equals_single_search(cabi):
    """SURVEY.md section 8(e): row-sharded search + merge is bit-identical to the single-shard search."""
    N, D, C, B, k, G = 40_000, 768, 20, 16, 5, 4
    P, _ = _synthetic_index(N, D, C)
    Q, _ = _synthetic_index(B, D, C, seed=1)
    Pg, Qg = P.cuda(), Q.cuda()
    d0, i0 = cabi.knn_l2_topk(Qg, Pg, k, algo=cabi.AC_KNN_EXACT)
    ds, is_ = [], []
    for g in range(G):
        lo, hi = g * N // G, (g + 1) * N // G
        d, i = cabi.knn_l2_topk(Qg, Pg[lo:hi].contiguous(), k, row_offset=lo, algo=cabi.AC_KNN_AUTO)
        ds.append(d); is_.append(i)
    dm, im = cabi.topk_merge(torch.stack(ds), torch.stack(is_))
    assert torch.equal(im, i0) and torch.equal(dm, d0)


def test_segment_mean(cabi):
    g = torch.Generator().manual_seed(5)
    X = torch.randn(200, 64, generator=g)
    cls = torch.randint(0, 7, (200,), generator=g)
    mean, cnt = cabi.segment_mean(X.cuda(), cls.cuda(), 8)
    for c in range(8):
        rows = X[cls == c]
        assert int(cnt[c]) == rows.shape[0]
        if rows.shape[0]:
            assert (mean[c].cpu() - torch.stack(list(rows)).mean(0)).abs().max() < 1e-6
        else:
            assert float(mean[c].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ head
def _head(D, C, dev="cuda"):
    p = ho.init_head(D, C)
    return p, {k: v.clone().to(dev).contiguous() for k, v in p.items()}


@pytest.mark.parametrize("B,D,C", [(1, 768, 20), (32, 768, 20), (257, 768, 1000), (5, 64, 3)])
def test_head_forward(cabi, B, D, C):
    p, pg = _head(D, C)
    X = torch.nn.functional.normalize(torch.randn(B, D, generator=torch.Generator().manual_seed(B)), dim=1)
    for act, name in ((cabi.AC_ACT_LOGITS, "logits"), (cabi.AC_ACT_SOFTMAX, "softmax"), (cabi.AC_ACT_SIGMOID, "sigmoid")):
        ref = ho.head_forward(X, p, name)
        out = cabi.head_forward(X.cuda(), pg, act).cpu()
        assert (out - ref).abs().max() < 1e-5, name       # north_star: logits within 1e-3


@pytest.mark.parametrize("loss_kind", ["ce", "bce"])
def test_head_train_steps_match_oracle(cabi, loss_kind):
    """3 optimizer steps (fwd with injected dropout masks, loss, bwd, clip, AdamW) vs the torch-CPU restatement.
    ReLU'(a) is discontinuous at a = 0: a batch with a pre-activation within fp32 summation noise of zero (seed 9 of an
    earlier version of this test had a1[19,33] = -9e-9) makes GPU and CPU legitimately disagree on a whole gradient
    row, so batches are drawn until every |pre-activation| > 1e-6."""
    B, D, C = 32, 768, 20
    g = torch.Generator().manual_seed(9)
    p, pg = _head(D, C)
    m = {k: torch.zeros_like(v) for k, v in p.items()}
    v = {k: torch.zeros_like(v2) for k, v2 in p.items()}
    mg = {k: torch.zeros_like(t) for k, t in pg.items()}
    vg = {k: torch.zeros_like(t) for k, t in pg.items()}
    for step in range(1, 4):
        while True:
            X = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
            masks = tuple(((torch.rand(B, n, generator=g) >= 0.1).float() / 0.9) for n in (D, D // 2))
            a0 = X @ p["W0"].t() + p["b0"]
            a1 = (torch.relu(a0) * masks[0]) @ p["W1"].t() + p["b1"]
            if min(a0.abs().min().item(), a1.abs().min().item()) > 1e-6:
                break
        if loss_kind == "ce":
            y = torch.randint(0, C, (B,), generator=g)
        else:
            y = (torch.rand(B, C, generator=g) < 0.2).float()
        loss_ref, grads, _ = ho.head_grads(X, y, p, masks, loss_kind)
        norm_ref = ho.clip_and_adamw(p, grads, m, v, step)
        stats = cabi.head_train_step(X.cuda(), y.cuda(), pg, mg, vg, step=step,
                                     loss_kind=cabi.AC_LOSS_CE if loss_kind == "ce" else cabi.AC_LOSS_BCE,
                                     masks=(masks[0].cuda(), masks[1].cuda())).cpu()
        assert abs(stats[0].item() - loss_ref.item()) < 1e-5
        assert abs(stats[2].item() - norm_ref.item()) < 1e-4 * max(1.0, norm_ref.item())
        for k in ho.PARAM_ORDER:
            diff = (pg[k].cpu() - p[k]).abs()
            # Adam's first steps move a weight by lr*sign(g): where |g| is at rounding level the sign is
            # ill-conditioned, so those (rare) elements may differ by up to 2*lr; everything else is tight
            solid = grads[k].abs() > 1e-6 * grads[k].abs().max()
            assert diff[solid].max() < 2e-5, (step, k, float(diff[solid].max()))
            assert diff.max() <= 2.1e-3 * step, (step, k)
            assert (mg[k].cpu() - m[k]).abs().max() <= 1e-6 + 1e-4 * m[k].abs().max(), (step, k)


def test_head_train_epoch_equals_step_sequence(cabi):
    """ac_head_train_epoch (device-side batch gather, all steps launched from C) == the same steps issued one by one"""
    n, D, C, bs = 100, 768, 7, 32
    g = torch.Generator().manual_seed(2)
    X = torch.nn.functional.normalize(torch.randn(n, D, generator=g), dim=1).cuda()
    y = torch.randint(0, C, (n,), generator=g).cuda()
    perm = torch.randperm(n, generator=g)
    _, pa = _head(D, C)
    pb = {k: v.clone() for k, v in pa.items()}
    ma, va = ({k: torch.zeros_like(v) for k, v in pa.items()} for _ in range(2))
    mb, vb = ({k: torch.zeros_like(v) for k, v in pb.items()} for _ in range(2))
    acc, nb = cabi.head_train_epoch(X, y, perm, pa, ma, va, first_step=5, batch=bs, seed=77)
    assert nb == 4
    tot = 0.0
    for b in range(nb):
        idx = perm[b * bs:(b + 1) * bs].cuda()
        st = cabi.head_train_step(X[idx].contiguous(), y[idx].contiguous(), pb, mb, vb, step=5 + b, seed=77)
        tot += float(st[0] + st[1])
    for k in pa:
        assert torch.equal(pa[k], pb[k]) and torch.equal(ma[k], mb[k]) and torch.equal(va[k], vb[k]), k
    assert abs(float(acc) - tot) < 1e-5


def test_ewc_penalty_and_fisher(cabi):
    B, D, C = 20, 768, 6
    g = torch.Generator().manual_seed(4)
    p, pg = _head(D, C)
    X = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    sampled = torch.randint(0, C, (B,), generator=g)
    fisher = {k: torch.zeros_like(v) for k, v in p.items()}
    ho.fisher_batch(X, sampled, p, 2, fisher)
    fg = {k: torch.zeros_like(t) for k, t in pg.items()}
    cabi.head_grad(X.cuda(), sampled.cuda(), pg, fisher=fg, inv_n_batches=0.5)
    for k in ho.PARAM_ORDER:
        assert (fg[k].cpu() - fisher[k]).abs().max() <= 1e-6 + 1e-4 * fisher[k].abs().max()
    # tests/test_ewc.py:128-153 of the reference: penalty > 0 after param += 0.1 and depends on batch_size
    star = {k: v.clone() for k, v in pg.items()}
    moved = {k: (v + 0.1).contiguous() for k, v in pg.items()}
    pen, _ = ho.ewc_penalty({k: v.cpu() for k, v in moved.items()}, fisher, p, 100.0, None)
    out = cabi.ewc_penalty(moved, fg, star, 100.0, None)
    assert out.item() > 0 and abs(out.item() - pen.item()) <= 1e-4 * pen.item()
    out32 = cabi.ewc_penalty(moved, fg, star, 100.0, 32)
    assert abs(out32.item() * 32 - out.item()) <= 1e-4 * out.item()


# ------------------------------------------------------------------------------------------------ encoder
def _small_bert(layers=2):
    sd, cfg, hf = eo.make_bert_state_dict(1234, num_hidden_layers=layers)
    return sd, cfg


def _encoder(cabi, sd, cfg, max_tokens, cls_only=True, arch="bert"):
    return cabi.Encoder(sd, arch=arch, layers=cfg.num_hidden_layers, hidden=cfg.hidden_size,
                        heads=cfg.num_attention_heads, intermediate=cfg.intermediate_size, vocab=cfg.vocab_size,
                        max_pos=cfg.max_position_embeddings, type_vocab=cfg.type_vocab_size,
                        ln_eps=cfg.layer_norm_eps, pad_idx=(cfg.pad_token_id or 0), max_tokens=max_tokens,
                        cls_only=cls_only)


@pytest.mark.parametrize("B,S,pad", [(2, 300, True), (3, 129, False), (1, 512, False), (2, 384, True)])
def test_encoder_long_sequences(cabi, B, S, pad):
    """128 < S <= 512 (the reference truncates at max_length = 512, classifier.py:1261): two-pass key-block attention"""
    sd, cfg = _small_bert(2)
    ids = eo.synthetic_ids(B, S)
    mask = torch.ones_like(ids)
    if pad:
        for b in range(B):
            n = S - 37 * (b + 1)
            mask[b, n:] = 0
            ids[b, n:] = 0
    ref = eo.encoder_forward_cls(sd, ids, mask)
    enc = _encoder(cabi, sd, cfg, max_tokens=B * S)
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    assert (out - ref).norm(dim=1).max() < 1e-3, (out - ref).norm(dim=1).max()
    enc.close()


def test_encoder_full_last_layer_and_hidden_state(cabi):
    """cls_only = 0 keeps the whole last hidden state (HF last_hidden_state) and gives the same CLS rows"""
    sd, cfg = _small_bert(2)
    B, S = 3, 64
    ids = eo.synthetic_ids(B, S)
    ref_cls, ref_hidden = eo.encoder_forward_cls(sd, ids, None, return_hidden=True)
    enc_full = _encoder(cabi, sd, cfg, B * S, cls_only=False)
    enc_cls = _encoder(cabi, sd, cfg, B * S, cls_only=True)
    a = enc_full.forward_cls(ids.to(torch.int32).cuda()).cpu()
    hid = enc_full.last_hidden(B, S).cpu().view(B, S, -1)
    b = enc_cls.forward_cls(ids.to(torch.int32).cuda()).cpu()
    assert (a - ref_cls).norm(dim=1).max() < 1e-3 and (b - ref_cls).norm(dim=1).max() < 1e-3
    assert (a - b).abs().max() < 1e-4            # CLS-only tail: LayerNorm materialised on B rows; full flow: deferred into the epilogues
    # per row: the CLS rows above carry the same fp16 operand rounding (||dq|| <= 2.5e-4 at 2 layers, precision study), and
    # every other row goes through the same GEMMs and attention
    rel = ((hid - ref_hidden).norm(dim=-1) / ref_hidden.norm(dim=-1)).max().item()
    print(f"full hidden state: max row rel err {rel:.3e}")
    assert rel < 1e-3, rel
    with pytest.raises(cabi.AdaptiveB200Error):
        enc_cls.last_hidden(B, S)
    enc_full.close(); enc_cls.close()


def test_encoder_distilbert(cabi):
    """DistilBERT (the encoder of the reference's examples/basic_usage.py:9) through Encoder.from_hf vs HF itself on CPU"""
    from transformers import DistilBertConfig, DistilBertModel
    torch.manual_seed(3)
    cfg = DistilBertConfig(vocab_size=400, dim=128, n_heads=2, n_layers=2, hidden_dim=256, max_position_embeddings=64)
    m = DistilBertModel(cfg).eval()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "LayerNorm" in n or "layer_norm" in n or n.endswith(".bias"):
                p.add_(0.1 * torch.randn(p.shape))
    ids = eo.synthetic_ids(5, 40, vocab=400)
    mask = torch.ones_like(ids)
    mask[1, 30:] = 0
    mask[4, 11:] = 0
    with torch.no_grad():
        ref = torch.nn.functional.normalize(m(input_ids=ids, attention_mask=mask).last_hidden_state[:, 0, :], dim=1)
    enc = cabi.Encoder.from_hf(m, max_tokens=5 * 40)
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    assert (out - ref).norm(dim=1).max() < 1e-3
    enc.close()


def test_encoder_roberta_positions_and_padding(cabi):
    """RoBERTa position ids (cumsum of non-pad + pad_idx, HF modeling_roberta.py:146-159), hidden 128 / 2 heads"""
    sd, cfg, _ = eo.make_bert_state_dict(5, arch="roberta", num_hidden_layers=2, hidden_size=128, num_attention_heads=2,
                                         intermediate_size=256, vocab_size=300, max_position_embeddings=130)
    B, S = 4, 40
    ids = eo.synthetic_ids(B, S, vocab=300, arch="roberta")
    for b in range(B):
        ids[b, S - 3 * b:] = 1
    mask = (ids != 1).long()
    ref = eo.encoder_forward_cls(sd, ids, mask, arch="roberta", num_heads=2, ln_eps=cfg.layer_norm_eps, pad_idx=1)
    enc = _encoder(cabi, sd, cfg, B * S, arch="roberta")
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    assert (out - ref).norm(dim=1).max() < 1e-3
    enc.close()


@pytest.mark.parametrize("layers,B,S,pad", [(1, 2, 128, False), (2, 3, 16, True), (12, 8, 128, False), (2, 5, 77, True)])
def test_encoder_cls_matches_oracle(cabi, layers, B, S, pad):
    """north_star tolerance: distances within 1e-3 <=> ||dq|| < 5e-4; measured budget for tf32(RNE) operands
    is 1.6e-4 on distances (oracle/precision_study.py)."""
    sd, cfg = _small_bert(layers)
    ids = eo.synthetic_ids(B, S)
    mask = torch.ones_like(ids)
    if pad:
        for b in range(B):
            n = S - 1 - 2 * b
            mask[b, n:] = 0
            ids[b, n:] = 0
    ref = eo.encoder_forward_cls(sd, ids, mask)
    enc = _encoder(cabi, sd, cfg, max_tokens=B * S)
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    e = (out - ref)
    assert e.abs().max() < 2e-4, e.abs().max()
    assert e.norm(dim=1).max() < 1e-3            # precision study: 5.7e-4 at 12 layers (fp16 == tf32 mantissa)
    P = torch.nn.functional.normalize(torch.randn(2048, out.shape[1], generator=torch.Generator().manual_seed(0)), dim=1)
    dd = (((out[:, None, :] - P[None]) ** 2).sum(-1) - ((ref[:, None, :] - P[None]) ** 2).sum(-1)).abs().max()
    assert dd < 1e-3, dd                        # the north_star tolerance itself (distances within 1e-3)
    assert (out.norm(dim=1) - 1).abs().max() < 1e-5
    enc.close()


def _perturb_layernorms(sd, seed=5):
    """random init has gamma = 1, beta = 0 and row means ~ 0, which would hide the rank-1 corrections of the deferred-LayerNorm
    epilogues (r (acc - mu c1) + c0 with gamma folded into the weights)"""
    g = torch.Generator().manual_seed(seed)
    for k in list(sd.keys()):
        if k.endswith("LayerNorm.weight"):
            sd[k] = 1.0 + 0.3 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("LayerNorm.bias"):
            sd[k] = 0.2 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("output.dense.bias"):
            sd[k] = sd[k] + 0.5
    return sd


@pytest.mark.parametrize("layers,B,S,cls_only,pad", [(2, 8, 128, True, False), (3, 5, 96, False, True), (12, 4, 128, True, False),
                                                      (2, 3, 300, True, True)])
def test_encoder_with_nontrivial_layernorms_matches_oracle(cabi, layers, B, S, cls_only, pad):
    """non-unit gamma (up to 1.9), non-zero beta and shifted row means: every term of the deferred LayerNorm is exercised"""
    sd, cfg, _ = eo.make_bert_state_dict(1234, num_hidden_layers=layers)
    sd = _perturb_layernorms(sd)
    ids = eo.synthetic_ids(B, S)
    mask = torch.ones_like(ids)
    if pad:
        for b in range(B):
            n = S - 1 - 2 * b
            mask[b, n:] = 0
            ids[b, n:] = 0
    ref, ref_hidden = eo.encoder_forward_cls(sd, ids, mask, return_hidden=True)
    enc = _encoder(cabi, sd, cfg, max_tokens=B * S, cls_only=cls_only)
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    e = out - ref
    assert e.abs().max() < 3e-4 and e.norm(dim=1).max() < 1e-3, (e.abs().max(), e.norm(dim=1).max())
    assert (out.norm(dim=1) - 1).abs().max() < 1e-5
    if not cls_only:
        hidden = enc.last_hidden(B, S).cpu()
        keep = mask.bool()
        d = hidden.view(B, S, -1)[keep] - ref_hidden[keep]
        rel = (d.norm(dim=-1) / ref_hidden[keep].norm(dim=-1)).max().item()
        print(f"nontrivial LayerNorms, full hidden state: max row rel err {rel:.3e}")
        assert rel < 1e-3, rel                   # per valid row, as the CLS rows above (||dq|| < 1e-3)
    enc.close()


def test_encoder_at_the_benched_batch_matches_oracle_on_sampled_rows(cabi):
    """BASELINE configs[2]: bert-base, B = 512 x S = 128 (65 536 tokens through every GEMM tile of the step bench.py times);
    8 sampled sequences against the fp32 CPU oracle"""
    sd, cfg = _small_bert(12)
    B, S = 512, 128
    ids = eo.synthetic_ids(B, S)
    enc = _encoder(cabi, sd, cfg, max_tokens=B * S)
    out = enc.forward_cls(ids.to(torch.int32).cuda()).cpu()
    sel = torch.tensor([0, 1, 63, 127, 128, 300, 510, 511])
    ref = eo.encoder_forward_cls(sd, ids[sel], None)
    e = out[sel] - ref
    assert e.norm(dim=1).max() < 1e-3 and e.abs().max() < 2e-4, (e.norm(dim=1).max(), e.abs().max())
    assert (out.norm(dim=1) - 1).abs().max() < 1e-5 and bool(torch.isfinite(out).all())
    enc.close()


def test_encoder_roberta_large_shape_with_real_position_ids(cabi):
    """BASELINE configs[4]: RoBERTa-large (24 layers x 1024, 16 heads, vocab 50265, type_vocab 1, eps 1e-5, pad_idx 1,
    position ids = cumsum(non-pad) + 1 -- HF models/roberta/modeling_roberta.py:146-159) with padded sequences"""
    sd, cfg, _ = eo.make_bert_state_dict(1234, arch="roberta", num_hidden_layers=24, hidden_size=1024, num_attention_heads=16,
                                         intermediate_size=4096, vocab_size=50265, max_position_embeddings=514, type_vocab_size=1,
                                         layer_norm_eps=1e-5, pad_token_id=1)
    B, S = 3, 128
    ids = eo.synthetic_ids(B, S, vocab=50265, arch="roberta")
    ids[1, 100:] = 1
    ids[2, 17:] = 1
    mask = (ids != 1).long()
    ref = eo.encoder_forward_cls(sd, ids, mask, arch="roberta", num_heads=16, ln_eps=cfg.layer_norm_eps, pad_idx=1)
    enc = _encoder(cabi, sd, cfg, B * S, arch="roberta")
    out = enc.forward_cls(ids.to(torch.int32).cuda(), mask.to(torch.int32).cuda()).cpu()
    e = out - ref
    assert e.norm(dim=1).max() < 1.5e-3, e.norm(dim=1).max()          # 24 layers of fp16-operand rounding (12 layers: 6e-4)
    P = torch.nn.functional.normalize(torch.randn(1024, 1024, generator=torch.Generator().manual_seed(0)), dim=1)
    dd = (((out[:, None, :] - P[None]) ** 2).sum(-1) - ((ref[:, None, :] - P[None]) ** 2).sum(-1)).abs().max()
    assert dd < 1e-3, dd                                               # the north_star tolerance (distances within 1e-3)
    enc.close()


def test_pipeline_device_and_host_boundaries(cabi):
    """E -> K -> class scores -> H -> blend through the pipeline handle == the same stages called one by one;
    device-buffer and host-buffer entry points agree bit for bit."""
    sd, cfg = _small_bert(2)
    B, S, N, D, C, k = 16, 128, 5000, 768, 20, 5
    P, _ = _synthetic_index(N, D, C)
    Pg = P.cuda()
    enc = _encoder(cabi, sd, cfg, max_tokens=B * S)
    ids = eo.synthetic_ids(B, S).to(torch.int32)
    p, pg = _head(D, C)
    row_class = (torch.arange(N) % C).to(torch.int32).cuda()
    pl = cabi.Pipeline(enc, Pg, B, S, k, head=pg, row_class=row_class)
    oc, osc = pl.predict_device(ids.cuda())
    oc, osc = oc.clone(), osc.clone()
    oc_h, osc_h = pl.predict_host(ids.pin_memory())
    assert torch.equal(oc.cpu(), oc_h) and torch.equal(osc.cpu(), osc_h)
    emb, kd, ki = pl.debug_views(B)
    emb2 = enc.forward_cls(ids.cuda())
    d2, i2 = cabi.knn_l2_topk(emb2, Pg, k)
    assert torch.equal(emb, emb2) and torch.equal(ki, i2) and torch.equal(kd, d2)
    # host restatement of classifier.py:1358-1384 on the device intermediates
    pc, ps = cabi.proto_class_scores(kd, ki, row_class)
    probs = cabi.head_forward(emb, pg, cabi.AC_ACT_SOFTMAX)
    hv, hi = cabi.topk_desc(probs, k)
    tv, ti = torch.topk(probs, k, dim=1)
    assert torch.equal(hv, tv)
    pc, ps, hv, hi = pc.cpu(), ps.cpu(), hv.cpu(), hi.cpu()
    for b in range(B):
        comb = {}
        for c, s_ in zip(pc[b].tolist(), ps[b].tolist()):
            if c >= 0:
                comb[c] = s_ * 0.7
        for v, j in zip(hv[b].tolist(), hi[b].tolist()):
            comb[j] = comb.get(j, 0) + v * 0.3
        pr = sorted(comb.items(), key=lambda x: x[1], reverse=True)
        tot = sum(v for _, v in pr)
        pr = [(c, v / tot) for c, v in pr][:k]
        assert [c for c, _ in pr] == oc[b].tolist()[: len(pr)]
        assert np.allclose([v for _, v in pr], osc[b].tolist()[: len(pr)], atol=1e-6)
    pl.close(); enc.close()


def test_pipeline_host_step_replayed_as_a_cuda_graph_equals_the_eager_step(cabi):
    """ac_pipeline_predict_host: first call with a batch size runs the ordinary launches, the second records the device part of
    the step as a CUDA graph, later calls replay it.  Every call gets different ids: the replays must read the staging buffer, not
    data baked in at capture time, must equal the device-boundary (always eager) result bit for bit, and must account for the same
    number of kernel launches; another batch size gets its own graph."""
    sd, cfg = _small_bert(2)
    Bmax, S, N, D, C, k = 8, 32, 3000, 768, 20, 5
    P, _ = _synthetic_index(N, D, C)
    Pg = P.cuda()
    enc = _encoder(cabi, sd, cfg, max_tokens=Bmax * S)
    p, pg = _head(D, C)
    row_class = (torch.arange(N) % C).to(torch.int32).cuda()
    pl = cabi.Pipeline(enc, Pg, Bmax, S, k, head=pg, row_class=row_class)
    per_call = {}
    for rep, B in enumerate([3, 3, 3, 3, 8, 8, 8, 3, 1, 1, 1]):
        ids = eo.synthetic_ids(B, S, seed=100 + rep).to(torch.int32)
        n0 = cabi.launch_count()
        oc_h, osc_h = pl.predict_host(ids.pin_memory())
        oc_h, osc_h = oc_h.clone(), osc_h.clone()
        n1 = cabi.launch_count()
        oc, osc = pl.predict_device(ids.cuda())
        torch.cuda.synchronize()
        n2 = cabi.launch_count()
        assert torch.equal(oc.cpu(), oc_h) and torch.equal(osc.cpu(), osc_h), (rep, B)
        assert n1 - n0 == n2 - n1 > 0, (rep, B, n1 - n0, n2 - n1)      # a replay accounts for the kernels it launches
        per_call.setdefault(B, []).append(n1 - n0)
    assert all(len(set(v)) == 1 for v in per_call.values())
    pl.close(); enc.close()


def test_proto_class_scores_reduces_to_reference_form(cabi):
    """one row per class (the reference's usage): ac_proto_class_scores == memory.py:117-134 (ac_proto_scores)"""
    rng = np.random.default_rng(1)
    d = np.sort(rng.uniform(0, 4, size=(9, 6)).astype(np.float32), axis=1)
    idx = np.stack([rng.permutation(50)[:6] for _ in range(9)]).astype(np.int64)
    dg, ig = torch.from_numpy(d).cuda(), torch.from_numpy(idx).cuda()
    cls, sc = cabi.proto_class_scores(dg, ig, None)
    assert torch.equal(cls.cpu().long(), torch.from_numpy(idx))
    assert np.abs(sc.cpu().numpy() - ko.proto_scores(d, idx)).max() < 1e-6
    # many rows per class: the nearest row of a class wins, later rows of the same class are dropped
    rc = torch.tensor([i % 3 for i in range(50)], dtype=torch.int32).cuda()
    cls2, sc2 = cabi.proto_class_scores(dg, ig, rc)
    for b in range(9):
        seen, exp = [], []
        for j in range(6):
            c = int(idx[b, j]) % 3
            if c not in seen:
                seen.append(c); exp.append(np.exp(-d[b, j]))
        e = np.exp(np.array(exp, dtype=np.float32) - max(exp)); e /= e.sum()
        assert cls2[b].tolist()[: len(seen)] == seen and cls2[b].tolist()[len(seen):] == [-1] * (6 - len(seen))
        assert np.abs(sc2[b].cpu().numpy()[: len(seen)] - e).max() < 1e-6
