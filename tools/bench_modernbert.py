"""Stage E of ModernBERT-base on one B200: ids -> unit CLS rows through ac_encoder_create_modernbert, against HF
ModernBertModel on the same card in the same process.

    python tools/bench_modernbert.py [--layers 22] [--B 512] [--S 128] [--steps 20] [--warmup 5] [--out FILE]

Seeded random-init ModernBERT-base (adaptive_classifier_b200.workload.modernbert_base_state_dict), synthetic ids (CLS 50281,
SEP 50282, ids in [1000, 50368), no padding).  Before timing, 8 sampled rows are checked against the fp32 oracle
(tests/modernbert_oracle.py).  Times are CUDA events over `steps` calls after `warmup` calls.  Achieved TFLOP/s use
algorithmic flops computed here: linear = 2 M (3 H^2 + H^2 + 2 H I + I H) per layer; attention = 4 B heads 64 sum_q keys(q),
keys(q) = S for global layers and |{k : |q - k| <= window}| for sliding ones.  Prints one JSON line (and writes it to --out).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def flops(dims, B, S):
    H, I, heads = dims["hidden"], dims["intermediate"], dims["heads"]
    M = B * S
    lin = dims["layers"] * 2.0 * M * (3 * H * H + H * H + 2 * H * I + I * H)
    att = 0.0
    for w in dims["windows"]:
        if w == 0:
            keys = S * S
        else:
            keys = sum(min(S - 1, q + w) - max(0, q - w) + 1 for q in range(S))
        att += 4.0 * B * heads * 64 * keys
    return lin, att


def time_fn(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=22)
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--S", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"

    from adaptive_classifier_b200 import _cabi, build, workload
    import modernbert_oracle as mo
    build.build_library()
    m, cfg = workload.modernbert_base_state_dict(1234, num_hidden_layers=a.layers)
    dims = _cabi.modernbert_dims(cfg)
    ids = workload.modernbert_synthetic_ids(a.B, a.S, vocab=cfg.vocab_size)
    ids_dev = ids.cuda()
    enc = _cabi.Encoder.from_hf(m, max_tokens=a.B * a.S)
    out = torch.empty((a.B, cfg.hidden_size), dtype=torch.float32, device="cuda")

    # correctness before timing: 8 sampled rows against the fp32 oracle
    enc.forward_cls(ids_dev, out=out)
    rows = torch.linspace(0, a.B - 1, 8).long()
    sd = {k: v.detach().float() for k, v in m.state_dict().items()}
    want = mo.modernbert_forward_cls(sd, ids[rows].long(), None, cfg).double()
    got = out[rows.cuda()].double().cpu()
    dq = (got - want).norm(dim=1).max().item()
    assert dq < 1e-3, dq

    ms = time_fn(lambda: enc.forward_cls(ids_dev, out=out), a.steps, a.warmup)
    lin, att = flops(dims, a.B, a.S)

    # HF ModernBertModel on the same card: torch eager (sdpa attention) in TF32, and under fp16 autocast
    hf = m.cuda().eval()
    ids64 = ids_dev.long()
    mask = torch.ones_like(ids64)

    def hf_step():
        with torch.no_grad():
            h = hf(input_ids=ids64, attention_mask=mask).last_hidden_state[:, 0]
            return torch.nn.functional.normalize(h, dim=1)

    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    hf_tf32 = time_fn(hf_step, max(5, a.steps // 4), 2)

    def hf_fp16():
        with torch.autocast("cuda", dtype=torch.float16):
            return hf_step()

    hf_f16 = time_fn(hf_fp16, max(5, a.steps // 4), 2)
    res = {
        "workload": f"ModernBERT-base stage E (ids -> unit CLS rows), {a.layers} layers, B={a.B}, S={a.S}, seeded random init",
        "card": card(),
        "stage_e_ms": round(ms, 3),
        "tokens_per_s": round(a.B * a.S / ms * 1e3),
        "linear_tflops_algorithmic": round(lin / 1e12, 3),
        "attention_tflops_algorithmic": round(att / 1e12, 3),
        "achieved_tflop_s_total": round((lin + att) / ms / 1e9, 1),
        "hf_eager_tf32_ms": round(hf_tf32, 3),
        "hf_fp16_autocast_sdpa_ms": round(hf_f16, 3),
        "speedup_vs_hf_tf32": round(hf_tf32 / ms, 2),
        "speedup_vs_hf_fp16": round(hf_f16 / ms, 2),
        "max_l2_err_sampled_rows": dq,
        "steps": a.steps, "warmup": a.warmup,
        "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
    }
    # per-class kernel times over one profiled forward (GEMMs vs attention)
    _cabi.profile_enable(True)
    for c in (0, 1):
        _cabi.profile_read(c)
    enc.forward_cls(ids_dev, out=out)
    torch.cuda.synchronize()
    g, t = _cabi.profile_read(0), _cabi.profile_read(1)
    _cabi.profile_enable(False)
    res["gemm_ms_profiled"] = round(g["ms"], 3)
    res["attention_ms_profiled"] = round(t["ms"], 3)
    res["gemm_tflop_s"] = round(lin / g["ms"] / 1e9, 1) if g["ms"] > 0 else None
    res["attention_tflop_s"] = round(att / t["ms"] / 1e9, 1) if t["ms"] > 0 else None
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
