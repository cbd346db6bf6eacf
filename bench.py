#!/usr/bin/env python
"""bench.py -- queries/sec of predict() on the BASELINE.json workload (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A step = one predict pass (E encoder -> K prototype kNN -> H head -> blend, top-5 labels) over one batch of
512 synthetic 128-token queries PER GPU against a 1M x 768 fp32 prototype matrix (1000 classes), the
configuration BASELINE.json's metric is quoted on (configs[2]); it fits one B200, and at N > 1 the matrix is
row-sharded while every rank keeps its own 512 queries (weak scaling; --strong keeps the GLOBAL batch at 512).
One JSON line on rank 0.  Before the timed region the step's kNN result of 16 queries is checked against the CPU oracle
(and, at N > 1, the merged sharded result against the unsharded search): `parity_checked`.
At N = 1 the line also carries sub-results measured after the headline (never inside its timed region): `k_equals_C`
(predict() semantics, k = 1000), `cfg4` (BASELINE configs[3], the add_examples loop), `gpu_library_baseline` (HF BertModel in
torch eager on the same GPU) and `cpu_baseline` (the oracle port on the host cores).
--dump-outputs DIR writes what the last timed step returned (top-5 class ids and scores of every query of this rank) as
DIR/top5_classes.npy (float64) and DIR/top5_scores.npy (float32); at N > 1 each rank writes its own, suffixed _rank<r>.  Every
input is seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "queries/sec predict() bert-base 128-tok, 1M x 768 prototypes"
B_PER_GPU, S, D, N_ROWS, C, K_TOP = 512, 128, 768, 1_000_000, 1000, 5
WORKLOAD = ("bert-base-uncased architecture (random init seed 1234), S=128, batch 512/GPU, 1M x 768 fp32 prototypes, "
            "1000 classes, k=5 (predict_batch semantics), prototype rows sharded across GPUs")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"hbm_gbs": j["hbm_gbs"], "bf16_tflops": j["bf16_tflops"],
                "bf16_tflops_sustained": j.get("bf16_tflops_sustained", j["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx = float(f[2]); power.append(float(f[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's own path (HF BertModel CPU forward -> IndexFlatL2 restatement,
# nq = 1 per query as in memory.py:110 -> torch head -> blend), on this box's host cores.
# ------------------------------------------------------------------------------------------------
class CpuPath:
    def __init__(self, n_rows=N_ROWS):
        import numpy as np
        import torch
        from oracle import knn_oracle as ko
        from oracle import head_oracle as ho
        from adaptive_classifier_b200 import workload as wl
        self.torch, self.np, self.ko, self.ho = torch, np, ko, ho
        self.avail = len(os.sched_getaffinity(0))
        self.model, self.cfg = wl.bert_base_state_dict(1234)
        self.cores = self._calibrate_threads(torch, wl)
        self.P = wl.synthetic_rows(0, n_rows, D, C, seed=0, device="cpu").numpy()
        self.row_class = (np.arange(n_rows) % C).astype(np.int64)
        self.head = ho.init_head(D, C)
        ko.lib()
        self.wl = wl

    def _calibrate_threads(self, torch, wl):
        """'all the host threads it can use': the affinity mask of a container often exceeds its CPU quota, and an
        oversubscribed oneDNN pool is several times slower, so the encoder thread count is the fastest of a short
        sweep up to the affinity size."""
        ids = wl.synthetic_ids(8, S).to(torch.int64)
        best, best_t = 1, float("inf")
        cand = sorted({n for n in (4, 8, 16, 32, 64, self.avail) if n <= self.avail})
        for n in cand:
            torch.set_num_threads(n)
            with torch.no_grad():
                self.model(input_ids=ids[:2])
                t0 = time.time()
                self.model(input_ids=ids)
                dt = time.time() - t0
            if dt < best_t:
                best, best_t = n, dt
        torch.set_num_threads(best)
        return best

    def predict(self, ids):
        """ids int64 [q, S] -> list of top-5 (class, score); returns per-stage seconds too."""
        torch, np, ko, ho = self.torch, self.np, self.ko, self.ho
        from concurrent.futures import ThreadPoolExecutor
        t0 = time.time()
        with torch.no_grad():
            h = self.model(input_ids=ids, attention_mask=torch.ones_like(ids)).last_hidden_state[:, 0, :]
            emb = torch.nn.functional.normalize(h, p=2, dim=1)
        t1 = time.time()
        q = emb.numpy()

        def one(b):   # nq = 1 per call like the reference; ctypes releases the GIL
            return ko.knn_l2(q[b : b + 1], self.P, K_TOP)
        with ThreadPoolExecutor(max_workers=min(self.avail, 64)) as ex:
            res = list(ex.map(one, range(q.shape[0])))
        t2 = time.time()
        out = []
        probs = ho.head_forward(emb, self.head, "softmax")
        for b, (d, i) in enumerate(res):
            s = ko.proto_scores(d, i)[0]
            comb = {}
            for idx, sc in zip(i[0], s):
                c = int(self.row_class[idx])
                if c not in comb:
                    comb[c] = float(sc) * 0.7
            hv, hi = torch.topk(probs[b], K_TOP)
            for v, j in zip(hv.tolist(), hi.tolist()):
                comb[j] = comb.get(j, 0.0) + v * 0.3
            pr = sorted(comb.items(), key=lambda x: x[1], reverse=True)
            tot = sum(v for _, v in pr)
            out.append([(c, v / tot) for c, v in pr][:K_TOP])
        t3 = time.time()
        return out, {"encoder_s": t1 - t0, "knn_s": t2 - t1, "head_blend_s": t3 - t2}


def cpu_baseline(n_queries=32):
    import torch
    cp = CpuPath()
    ids = cp.wl.synthetic_ids(n_queries, S).to(torch.int64)
    cp.predict(ids)                                      # warm-up at the same shape (oneDNN primitives, page-in)
    t0 = time.time()
    _, stages = cp.predict(ids)
    dt = time.time() - t0
    return {"value": n_queries / dt, "unit": "queries/s", "cores": cp.cores, "kind": "port",
            "sample": (f"{n_queries} queries of the same workload: HF BertModel fp32 CPU forward ({cp.cores} threads = fastest of a "
                       f"sweep up to the {cp.avail}-CPU affinity mask), IndexFlatL2 restatement nq=1 per query over the full "
                       f"1M x 768 matrix (queries in parallel threads), torch head + blend; FAISS itself is unavailable offline, "
                       f"so top-k ids are exact modulo ~1e-7 near-ties of a real faiss build (FMA contraction)"),
            "stages_s": {k: round(v, 3) for k, v in stages.items()}}


def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    cp = CpuPath(args.rows or N_ROWS)
    cp.predict(cp.wl.synthetic_ids(8, S).to(torch.int64))
    t_probe0 = time.time()
    cp.predict(cp.wl.synthetic_ids(8, S).to(torch.int64))
    per_q = (time.time() - t_probe0) / 8
    budget = 150.0
    nq = int(max(1, min(32, budget / max(1e-3, per_q * (args.steps + args.warmup)))))
    ids = cp.wl.synthetic_ids(nq, S).to(torch.int64)
    for _ in range(args.warmup):
        cp.predict(ids)
    t0 = time.time()
    for _ in range(args.steps):
        cp.predict(ids)
    dt = time.time() - t0
    v = nq * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "queries_per_step": nq},
            "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cp.cores, "kind": "port",
                             "sample": f"{nq} queries per step, oracle port of the reference path on {cp.cores} host threads "
                                       "(HF CPU encoder + IndexFlatL2 restatement + torch head)"},
            "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# sub-results (N = 1, after the headline)
# ------------------------------------------------------------------------------------------------
def _timed_ms(torch, fn, steps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def sub_k_equals_c(torch, _cabi, enc, P, p_sqnorm, p_half, row_class, hp, ids_dev, steps):
    """predict() semantics (classifier.py:415-480) batched: k = num_classes nearest ROWS, one score per class (nearest row
    of the class), head softmax over all classes, per-class blend weights, renormalise, top-5 -- every stage on the device"""
    B = ids_dev.shape[0]
    stats = torch.zeros(4, dtype=torch.int32, device=ids_dev.device)
    wp = torch.full((C,), 0.7, device=ids_dev.device)       # training_history >= 10 for every class of the synthetic index
    wh = torch.full((C,), 0.3, device=ids_dev.device)

    def step():
        emb = enc.forward_cls(ids_dev)
        d, i = _cabi.knn_l2_topk(emb, P, C, p_sqnorm=p_sqnorm, p_half=p_half, stats=stats)
        pc, ps = _cabi.proto_class_scores(d, i, row_class, n_classes=C)
        probs = _cabi.head_forward(emb, hp, _cabi.AC_ACT_SOFTMAX)
        return _cabi.blend_dense(pc, ps, probs, wp, wh, K_TOP)

    ms = _timed_ms(torch, step, steps)
    emb = enc.forward_cls(ids_dev)
    ms_knn = _timed_ms(torch, lambda: _cabi.knn_l2_topk(emb, P, C, p_sqnorm=p_sqnorm, p_half=p_half, stats=stats), steps)
    ms_knn_exact8 = _timed_ms(torch, lambda: _cabi.knn_l2_topk(emb[:8], P, C, algo=_cabi.AC_KNN_EXACT), 2, warmup=1)
    # parity of the k = C search on 4 queries against the exact scan (bit-identical)
    d, i = _cabi.knn_l2_topk(emb, P, C, p_sqnorm=p_sqnorm, p_half=p_half, stats=stats)
    d0, i0 = _cabi.knn_l2_topk(emb[:4].contiguous(), P, C, algo=_cabi.AC_KNN_EXACT)
    ok = bool(torch.equal(i[:4], i0) and torch.equal(d[:4], d0))
    st = stats.cpu().tolist()
    return {"k": C, "queries_per_s": B / (ms * 1e-3), "ms_per_step": ms, "knn_ms": ms_knn, "knn_path": "tensor (two passes + exact re-rank)",
            "knn_exact_scan_ms_per_8_queries": ms_knn_exact8, "knn_equals_exact_scan": ok,
            "knn_overflow_queries": st[1], "knn_max_collected": st[2]}


def sub_gpu_library_baseline(torch, ids_dev, enc_ms):
    """stage E comparator of SURVEY 2b: the reference's own encoder call (HF BertModel, torch eager, SDPA) on the same B200"""
    from adaptive_classifier_b200 import workload as wl
    out = {}
    try:
        model, _ = wl.bert_base_state_dict(1234)
        model = model.cuda().eval()
        ids = ids_dev.long()
        mask = torch.ones_like(ids)

        def fwd():
            with torch.no_grad():
                return torch.nn.functional.normalize(model(input_ids=ids, attention_mask=mask).last_hidden_state[:, 0, :], dim=1)
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        out["hf_eager_fp32_ms"] = _timed_ms(torch, fwd, 2, warmup=1)
        torch.backends.cuda.matmul.allow_tf32 = True
        out["hf_eager_tf32_ms"] = _timed_ms(torch, fwd, 5, warmup=2)
        torch.backends.cuda.matmul.allow_tf32 = prev

        def fwd16():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
                return model(input_ids=ids, attention_mask=mask).last_hidden_state[:, 0, :]
        out["hf_eager_fp16_autocast_ms"] = _timed_ms(torch, fwd16, 5, warmup=2)
        out["this_encoder_ms"] = enc_ms
        out["queries_per_s"] = {k[:-3]: ids.shape[0] / (v * 1e-3) for k, v in out.items() if k.endswith("_ms")}
        out["note"] = ("stage E only (ids -> unit CLS rows) at B = 512 x S = 128; cuBLAS / SDPA library kernels of torch "
                       f"{torch.__version__}; fp16 autocast does not meet the 1e-3 distance tolerance by construction (fp16 residual stream)")
        del model
        torch.cuda.empty_cache()
    except Exception as ex:          # a context number must never take the headline down
        out["failed"] = repr(ex)
    return out


def sub_cfg4(examples):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_add_examples as bae
    return bae.run(examples=examples, call=256, seq=128, quiet=True)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg3", "cfg5"], help=argparse.SUPPRESS)
    ap.add_argument("--strong", action="store_true", help="strong scaling: the GLOBAL batch stays 512 (512 / N queries per GPU)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-results (k = C, cfg4, HF-eager comparator)")
    ap.add_argument("--cfg4-examples", type=int, default=50_000, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's top-5 class ids and scores as DIR/<name>.npy (B200 path only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the B200 path's outputs; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    # BASELINE.json configs[1] / [2] (default, the one the metric is quoted on) / [4]
    global B_PER_GPU, D, N_ROWS, C, WORKLOAD
    arch_over = {}
    if args.workload == "cfg2":
        B_PER_GPU, N_ROWS, C = 256, 100_000, 20
        WORKLOAD = "bert-base-uncased architecture, S=128, batch 256/GPU, 100k x 768 fp32 prototypes, 20 classes, k=5"
    elif args.workload == "cfg5":
        B_PER_GPU, N_ROWS, C, D = 128, 500_000, 50, 1024
        WORKLOAD = ("roberta-large architecture (24 x 1024, 16 heads, vocab 50265, RoBERTa position ids from pad_idx + 1, eps 1e-5; random "
                    "init), S=128, batch 128/GPU, 500k x 1024 fp32 prototypes, 50 labels, k=5 (multilabel predict(): sigmoid head + "
                    "prototype fallback share this device pass; thresholds are host logic)")
    if args.rows is None:
        args.rows = N_ROWS

    import torch
    import torch.distributed as dist
    from adaptive_classifier_b200 import _cabi, workload as wl
    from adaptive_classifier_b200.models import AdaptiveHead
    from adaptive_classifier_b200.parallel import ShardedPipeline, shard_bounds

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    _cabi.load_library()          # fails loudly if the in-tree .so is missing
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    G = world
    n_rows = args.rows
    Bq = B_PER_GPU // G if args.strong else B_PER_GPU                # queries of this rank per step
    if args.strong and B_PER_GPU % G:
        raise SystemExit("--strong needs the global batch to divide by the number of GPUs")

    # ---- build the replica: encoder + head (replicated), prototype shard
    if args.workload == "cfg5":
        from transformers import RobertaConfig, RobertaModel
        torch.manual_seed(1234)
        rc_cfg = RobertaConfig(vocab_size=50265, hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096,
                               max_position_embeddings=514, type_vocab_size=1, layer_norm_eps=1e-5, pad_token_id=1)
        model = RobertaModel(rc_cfg, add_pooling_layer=False).eval()
        vocab = 50265
    else:
        model, cfg = wl.bert_base_state_dict(1234, **arch_over)
        vocab = 30522
    enc = _cabi.Encoder.from_hf(model, max_tokens=max(Bq, 16) * S, device=dev)
    del model
    lo, hi = shard_bounds(n_rows, rank, G)
    P = wl.synthetic_rows(lo, hi, D, C, seed=0, device=dev)
    p_sqnorm = _cabi.row_sqnorm(P)
    p_half = _cabi.knn_make_shadow(P)          # index-build-time fp16 shadow for the tensor path's coarse pass
    row_class = (torch.arange(n_rows, device=dev) % C).to(torch.int32)
    head = AdaptiveHead(D, C, hidden_dims=[D, D // 2]).to(dev).eval()
    hp = head._param_dict()
    if args.workload == "cfg5":     # RoBERTa: <s> = 0 first, </s> = 2 last, never the pad id 1
        g = torch.Generator().manual_seed(7 + rank)
        ids_host = torch.randint(1000, vocab, (Bq, S), generator=g, dtype=torch.int64).to(torch.int32)
        ids_host[:, 0], ids_host[:, -1] = 0, 2
        ids_host = ids_host.pin_memory()
    else:
        ids_host = wl.synthetic_ids(Bq, S, seed=7 + rank).pin_memory()
    ids_dev = ids_host.to(dev)
    torch.cuda.synchronize()

    pipe = _cabi.Pipeline(enc, P, Bq, S, K_TOP, head=hp, row_class=row_class, p_sqnorm=p_sqnorm, p_half=p_half, row_offset=lo, shards=G)
    if G == 1:
        def step_device():
            return pipe.predict_device(ids_dev)

        def step_host():
            return pipe.predict_host(ids_host)
    else:
        sp = ShardedPipeline(pipe)
        out_cls_host = torch.empty((Bq, K_TOP), dtype=torch.int32).pin_memory()
        out_sc_host = torch.empty((Bq, K_TOP), dtype=torch.float32).pin_memory()
        ids_stage = torch.empty_like(ids_dev)

        def step_device():
            return sp.predict_device(ids_dev)

        def step_host():
            ids_stage.copy_(ids_host, non_blocking=True)
            oc, osc = sp.predict_device(ids_stage)
            out_cls_host.copy_(oc, non_blocking=True)
            out_sc_host.copy_(osc, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return out_cls_host, out_sc_host

    def barrier():
        if G > 1:
            dist.barrier()

    def timed(fn, steps):
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize(); barrier()
        t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if G > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1, out

    # ---- warm-up, shape sanity and the parity check of this very step (outside the timed region)
    for _ in range(args.warmup):
        oc, osc = step_device()
    torch.cuda.synchronize()
    assert oc.shape == (Bq, K_TOP) and bool((osc[:, 0] > 0).all()) and bool((oc[:, 0] >= 0).all())
    parity = {"parity_checked": False}
    emb, kd, ki = pipe.debug_views(Bq)          # unit CLS rows and the (merged) kNN result of the last step
    nchk = min(16, Bq)
    if G > 1:
        # the merged sharded result of rank 0's queries == the unsharded search over the whole matrix (bit-identical)
        ok_unsharded = True
        if rank == 0:
            Pfull = wl.synthetic_rows(0, n_rows, D, C, seed=0, device=dev)
            d_u, i_u = _cabi.knn_l2_topk(emb[:nchk].contiguous(), Pfull, K_TOP, algo=_cabi.AC_KNN_EXACT)
            ok_unsharded = bool(torch.equal(i_u, ki[:nchk]) and torch.equal(d_u, kd[:nchk]))
            del Pfull
            torch.cuda.empty_cache()
        parity["sharded_equals_unsharded_search"] = ok_unsharded
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import knn_oracle as ko     # the checker, outside every timed region
        Pcpu = wl.synthetic_rows(0, n_rows, D, C, seed=0, device=dev).cpu().numpy() if G > 1 else P.cpu().numpy()
        d_ref, i_ref = ko.knn_l2(emb[:nchk].cpu().numpy(), Pcpu, K_TOP)
        import numpy as np
        ok = bool(np.array_equal(ki[:nchk].cpu().numpy(), i_ref) and np.array_equal(kd[:nchk].cpu().numpy(), d_ref))
        del Pcpu
        parity.update({"parity_checked": True, "knn_top5_equals_oracle": ok, "queries_checked": nchk,
                       "note": "ids and distances bit-identical to oracle/knn_oracle.c (IndexFlatL2 restatement; real FAISS is "
                               "unavailable offline: exact modulo ~1e-7 near-ties of an FMA-contracting faiss build)"})
        if not ok or not parity.get("sharded_equals_unsharded_search", True):
            raise SystemExit(f"bench.py: parity check failed: {parity}")
    pipe.knn_stats(reset=True)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    _cabi.profile_enable(True)
    l0 = _cabi.launch_count()
    ms, t0, t1, last = timed(step_device, args.steps)
    launches = _cabi.launch_count() - l0
    _cabi.profile_enable(False)
    prof = {c: _cabi.profile_read(c) for c in range(5)}
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    kstats = pipe.knn_stats(reset=True)
    if args.dump_outputs:
        # copied before anything else runs: the step returns views of the pipeline's output buffers
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        sfx = f"_rank{rank}" if G > 1 else ""
        np.save(os.path.join(args.dump_outputs, f"top5_classes{sfx}.npy"), last[0].cpu().numpy().astype(np.float64))
        np.save(os.path.join(args.dump_outputs, f"top5_scores{sfx}.npy"), last[1].cpu().numpy().astype(np.float32))
    for _ in range(2):
        step_host()
    ms_e2e, _, _, _ = timed(step_host, args.steps)
    # the scan kernel by itself (same queries, same shard, nothing else on the GPU): inside the step it shares the SMs with the head
    # forward on the side stream, which is what `ms_per_launch` above includes
    knn_alone_ms = None
    if rank == 0:
        q_alone = emb.repeat(G, 1).contiguous() if G > 1 else emb.contiguous()
        kw = dict(p_sqnorm=p_sqnorm, p_half=p_half)
        for _ in range(2):
            _cabi.knn_l2_topk(q_alone, P, K_TOP, **kw)
        torch.cuda.synchronize()
        _cabi.profile_enable(True)
        for _ in range(5):
            _cabi.knn_l2_topk(q_alone, P, K_TOP, **kw)
        _cabi.profile_enable(False)
        pa = _cabi.profile_read(2)
        knn_alone_ms = pa["ms"] / max(1, pa["launches"])

    if rank != 0:
        if G > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    total_q = G * Bq * args.steps
    value = total_q / (ms / 1e3)
    gemm, att, knn, knn2 = prof[0], prof[1], prof[2], prof[4]
    gemm_tflops = gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 if gemm["ms"] > 0 else 0.0
    n_local = hi - lo
    q_scan = G * Bq                                             # queries every rank scans its shard for
    knn_ms = knn["ms"] / max(1, knn["launches"])
    knn_alg_gbs = 4.0 * n_local * D / (knn_ms * 1e-3) / 1e9 if knn_ms > 0 else 0.0
    knn_streamed_bytes = 2.0 * n_local * D + 4.0 * n_local + 2.0 * q_scan * D      # fp16 shadow + ||p||^2 + fp16 queries
    knn_str_gbs = knn_streamed_bytes / (knn_ms * 1e-3) / 1e9 if knn_ms > 0 else 0.0
    knn_tflops = 2.0 * q_scan * n_local * D / (knn_ms * 1e-3) / 1e12 if knn_ms > 0 else 0.0
    tfrac = knn_tflops / pk["bf16_tflops_sustained"]
    sfrac = knn_str_gbs / pk["hbm_gbs"]
    traffic_file = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    tj = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}
    line = {
        "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": G, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": G * Bq, "seq_len": S, "prototypes": n_rows,
                   "parallelism": f"dp{G} encoder/head, prototype rows sharded x{G}",
                   "exchange": "nccl: all-gather of unit embeddings + one packed all-to-all of (d, id) candidates" if G > 1 else "none",
                   "l2": "inputs larger than L2 every step (3.07 GB prototype matrix / G, ~2 GB activations per step)"},
        "e2e": {"value": total_q / (ms_e2e / 1e3), "unit": "queries/s",
                "h2d_bytes_per_step": Bq * S * 4 * G, "d2h_bytes_per_step": Bq * K_TOP * 8 * G,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity": parity,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel<Epi..., kind::f16> (encoder projections as CTA-pair tcgen05 GEMMs: fp16 operands, "
                                                  "fp32 TMEM accumulators, LayerNorm / GELU / residual fused into the epilogues)",
                     "achieved": gemm_tflops, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / pk["bf16_tflops_sustained"],
                     "traffic": tj.get("dram_bytes_per_launch"), "traffic_source": tj.get("source", "no ncu capture of this build committed"),
                     "peak_source": f"{pk['source']} cuBLAS bf16 GEMM, sustained (kernel timed inside a long step)",
                     "launches": gemm["launches"], "ms_total": gemm["ms"], "share_of_step": gemm["ms"] / ms},
        "roofline_knn": {"kernel": "gemm_tc_kernel<EpiKnn, kind::f16> (pass 1 of the prototype scan: tcgen05 coarse distances over the fp16 "
                                   "shadow, per-(query, CTA) top-16 lists)",
                         "ms_per_launch": knn_ms,
                         "frac_algorithmic": knn_alg_gbs / pk["hbm_gbs"], "algorithmic_gbs": knn_alg_gbs,
                         "algorithmic_bytes": "4*N*D: one read of the fp32 matrix (what IndexFlatL2 scans)",
                         "frac_streamed": sfrac, "streamed_gbs": knn_str_gbs,
                         "streamed_bytes": "2*N*D + 4*N + 2*B*D: what the kernel actually reads (fp16 shadow, ||p||^2, fp16 queries)",
                         "tensor_frac": tfrac, "tensor_tflops": knn_tflops,
                         "bound": "tensor" if tfrac >= sfrac else "hbm",
                         "peak_hbm_gbs": pk["hbm_gbs"], "peak_tflops": pk["bf16_tflops_sustained"], "peak_source": pk["source"],
                         "share_of_step": knn["ms"] / ms,
                         "alone": None if not knn_alone_ms else {
                             "ms_per_launch": knn_alone_ms, "frac_algorithmic": 4.0 * n_local * D / (knn_alone_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                             "tensor_frac": 2.0 * q_scan * n_local * D / (knn_alone_ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                             "note": "the same launch timed with nothing else on the GPU (in the step the head forward runs beside it on the side stream)"},
                         "second_pass_ms_per_launch": knn2["ms"] / max(1, knn2["launches"])},
        "knn_uncertified": kstats["second_pass_queries"] / max(1, kstats["searches"]),
        "knn_overflow": kstats["overflow_queries"],
        "attention": {"tflops_algorithmic": att["flops"] / (att["ms"] * 1e-3) / 1e12 if att["ms"] > 0 else 0.0,
                      "ms_total": att["ms"], "us_per_layer": 1e3 * att["ms"] / max(1, att["launches"]), "share_of_step": att["ms"] / ms},
    }
    if G == 1 and args.workload == "cfg3" and not args.no_extras:
        enc_ms = _timed_ms(torch, lambda: enc.forward_cls(ids_dev), 5)
        try:
            line["k_equals_C"] = sub_k_equals_c(torch, _cabi, enc, P, p_sqnorm, p_half, row_class, hp, ids_dev, 5)
        except Exception as ex:
            line["k_equals_C"] = {"failed": repr(ex)}
        line["gpu_library_baseline"] = sub_gpu_library_baseline(torch, ids_dev, enc_ms)
        del pipe
        del P, p_half, p_sqnorm
        torch.cuda.empty_cache()
        try:
            line["cfg4"] = sub_cfg4(args.cfg4_examples)
        except Exception as ex:
            line["cfg4"] = {"failed": repr(ex)}
    if G == 1 and not args.no_cpu_baseline and args.workload == "cfg3":
        try:
            line["cpu_baseline"] = cpu_baseline()
        except Exception as ex:           # the CPU arm must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "queries/s", "cores": len(os.sched_getaffinity(0)),
                                    "kind": "port", "sample": f"failed: {ex!r}"}
    print(json.dumps(line), flush=True)
    if G > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
