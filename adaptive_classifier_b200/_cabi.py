"""ctypes binding of libadaptive_b200.so (the C ABI declared in include/adaptive_b200.h).

This is the binding a maintainer of the reference would add (INTEGRATION.md).  PyTorch is used only for
device memory and streams: every call passes raw device pointers + the current CUDA stream.
There is NO CPU fallback: a missing library raises ImportError-like RuntimeError, a missing sm_100 device
makes every compute call raise AdaptiveB200Error.
"""
from __future__ import annotations

import ctypes
import threading
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libadaptive_b200.so")

AC_KNN_AUTO, AC_KNN_EXACT, AC_KNN_TENSOR = 0, 1, 2
AC_KNN_MAX_K = 2048
AC_KNN_TENSOR_MAX_K = 1024
AC_ACT_LOGITS, AC_ACT_SOFTMAX, AC_ACT_SIGMOID = 0, 1, 2
AC_LOSS_CE, AC_LOSS_BCE = 0, 1
AC_ARCH_BERT, AC_ARCH_ROBERTA, AC_ARCH_MODERNBERT = 0, 1, 2
AC_PREC_TF32, AC_PREC_F16 = 0, 1

EXPORTS = [
    "ac_version", "ac_last_error", "ac_device_check",
    "ac_knn_workspace_bytes", "ac_knn_l2_topk", "ac_knn_make_shadow", "ac_row_sqnorm", "ac_topk_merge", "ac_proto_scores",
    "ac_segment_mean", "ac_memory_append_prune",
    "ac_head_forward", "ac_head_train_workspace_bytes", "ac_head_train_step", "ac_head_train_epoch", "ac_head_phase_timing", "ac_head_train_plan", "ac_head_grad", "ac_ewc_penalty",
    "ac_encoder_create", "ac_encoder_create_modernbert", "ac_encoder_destroy", "ac_encoder_forward_cls", "ac_encoder_last_hidden", "ac_linear_tc", "ac_attention",
    "ac_proto_class_scores", "ac_proto_class_scores_n", "ac_blend_dense", "ac_topk_desc_workspace_bytes", "ac_topk_desc", "ac_blend_topk",
    "ac_pipeline_create", "ac_pipeline_destroy", "ac_pipeline_predict_device", "ac_pipeline_predict_host",
    "ac_pipeline_encode", "ac_pipeline_embeddings", "ac_pipeline_search_shard", "ac_pipeline_finish_sharded",
    "ac_pipeline_debug_copy", "ac_pipeline_knn_stats", "ac_launch_count", "ac_profile_enable", "ac_profile_read",
]


class AdaptiveB200Error(RuntimeError):
    pass


class HeadParams(Structure):
    _fields_ = [("D", c_int), ("H0", c_int), ("H1", c_int), ("C", c_int),
                ("W0", c_void_p), ("b0", c_void_p), ("W1", c_void_p), ("b1", c_void_p),
                ("W2", c_void_p), ("b2", c_void_p)]


class TrainCfg(Structure):
    _fields_ = [("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float),
                ("weight_decay", c_float), ("max_norm", c_float),
                ("step", c_int), ("loss_kind", c_int), ("dropout_p", c_float),
                ("mask0", c_void_p), ("mask1", c_void_p), ("seed", c_uint64),
                ("ewc_fisher", POINTER(HeadParams)), ("ewc_star", POINTER(HeadParams)),
                ("ewc_lambda", c_float), ("ewc_C_old", c_int)]


class EncoderConfig(Structure):
    _fields_ = [("arch", c_int), ("layers", c_int), ("hidden", c_int), ("heads", c_int), ("intermediate", c_int),
                ("vocab", c_int), ("max_pos", c_int), ("type_vocab", c_int), ("pad_idx", c_int),
                ("ln_eps", c_float), ("precision", c_int), ("max_tokens", c_int), ("cls_only", c_int)]


_PP = POINTER(c_void_p)


class EncoderWeights(Structure):
    _fields_ = [("word_emb", c_void_p), ("pos_emb", c_void_p), ("type_emb", c_void_p),
                ("emb_ln_w", c_void_p), ("emb_ln_b", c_void_p),
                ("q_w", _PP), ("q_b", _PP), ("k_w", _PP), ("k_b", _PP), ("v_w", _PP), ("v_b", _PP),
                ("ao_w", _PP), ("ao_b", _PP), ("ao_ln_w", _PP), ("ao_ln_b", _PP),
                ("ff1_w", _PP), ("ff1_b", _PP), ("ff2_w", _PP), ("ff2_b", _PP),
                ("out_ln_w", _PP), ("out_ln_b", _PP)]


class ModernBertEncoderConfig(Structure):
    _fields_ = [("layers", c_int), ("hidden", c_int), ("heads", c_int), ("intermediate", c_int), ("vocab", c_int),
                ("norm_eps", c_float), ("precision", c_int), ("max_tokens", c_int), ("cls_only", c_int),
                ("window", POINTER(c_int)), ("rope_theta", POINTER(c_float))]


class ModernBertEncoderWeights(Structure):
    _fields_ = [("tok_emb", c_void_p), ("emb_norm_w", c_void_p), ("emb_norm_b", c_void_p),
                ("attn_norm_w", _PP), ("attn_norm_b", _PP),
                ("Wqkv", _PP), ("Wqkv_b", _PP), ("Wo", _PP), ("Wo_b", _PP),
                ("mlp_norm_w", _PP), ("mlp_norm_b", _PP),
                ("Wi", _PP), ("Wi_b", _PP), ("mlp_Wo", _PP), ("mlp_Wo_b", _PP),
                ("final_norm_w", c_void_p), ("final_norm_b", c_void_p)]


_lib = None


def load_library() -> ctypes.CDLL:
    """Load the shared library and declare signatures.  Needs no GPU (symbol check only)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AdaptiveB200Error(
            f"{LIB_PATH} is missing: build it with `python -m adaptive_classifier_b200.build` "
            "(adaptive_classifier_b200 has no CPU or PyTorch fallback)")
    L = ctypes.CDLL(LIB_PATH)
    L.ac_version.restype = c_int
    L.ac_last_error.restype = c_char_p
    L.ac_device_check.restype = c_int
    L.ac_knn_workspace_bytes.argtypes = [c_int, c_int64, c_int, c_int, c_int, POINTER(c_size_t)]
    L.ac_knn_l2_topk.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p,
                                 c_int64, c_void_p, c_size_t, c_int, c_void_p, c_void_p]
    L.ac_knn_make_shadow.argtypes = [c_void_p, c_int64, c_int, c_void_p, c_void_p]
    L.ac_row_sqnorm.argtypes = [c_void_p, c_int64, c_int, c_void_p, c_void_p]
    L.ac_topk_merge.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_proto_scores.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]
    L.ac_segment_mean.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_memory_append_prune.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                         c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_head_forward.argtypes = [c_void_p, c_int, POINTER(HeadParams), c_int, c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_head_train_workspace_bytes.argtypes = [c_int, c_int, POINTER(HeadParams), POINTER(c_size_t)]
    L.ac_head_train_step.argtypes = [c_void_p, c_void_p, c_int, POINTER(HeadParams), POINTER(HeadParams),
                                     POINTER(HeadParams), POINTER(TrainCfg), c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_head_train_epoch.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, POINTER(HeadParams), POINTER(HeadParams),
                                      POINTER(HeadParams), POINTER(TrainCfg), c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_head_grad.argtypes = [c_void_p, c_void_p, c_int, POINTER(HeadParams), c_int, POINTER(HeadParams),
                               POINTER(HeadParams), c_float, c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_ewc_penalty.argtypes = [POINTER(HeadParams), POINTER(HeadParams), POINTER(HeadParams), c_float, c_float,
                                 c_int, c_void_p, c_void_p]
    L.ac_encoder_create.argtypes = [POINTER(EncoderConfig), POINTER(EncoderWeights), POINTER(c_void_p)]
    L.ac_encoder_create_modernbert.argtypes = [POINTER(ModernBertEncoderConfig), POINTER(ModernBertEncoderWeights), POINTER(c_void_p)]
    L.ac_encoder_destroy.argtypes = [c_void_p]
    L.ac_encoder_forward_cls.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]
    L.ac_encoder_last_hidden.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    L.ac_linear_tc.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                               c_int, c_int, c_void_p]
    L.ac_attention.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    L.ac_proto_class_scores.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_proto_class_scores_n.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_blend_dense.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_topk_desc_workspace_bytes.argtypes = [c_int, c_int, c_int, POINTER(c_size_t)]
    L.ac_topk_desc.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    L.ac_blend_topk.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float,
                                c_void_p, c_void_p, c_void_p]
    L.ac_pipeline_create.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, POINTER(HeadParams),
                                     c_int, c_int, c_int, c_int64, c_int, POINTER(c_void_p)]
    L.ac_pipeline_encode.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p]
    L.ac_pipeline_embeddings.argtypes = [c_void_p, POINTER(c_void_p)]
    L.ac_pipeline_search_shard.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]
    L.ac_pipeline_finish_sharded.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_pipeline_destroy.argtypes = [c_void_p]
    L.ac_pipeline_predict_device.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_pipeline_predict_host.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    L.ac_pipeline_debug_copy.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    L.ac_profile_enable.argtypes = [c_int]
    L.ac_pipeline_knn_stats.argtypes = [c_void_p, c_void_p, c_int, c_void_p]
    L.ac_profile_read.argtypes = [c_int, POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(ctypes.c_double),
                                  POINTER(ctypes.c_longlong)]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name == "ac_launch_count":
            fn.restype = ctypes.c_longlong
        elif name not in ("ac_last_error",):
            fn.restype = c_int
    _lib = L
    return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load_library().ac_last_error()
        raise AdaptiveB200Error(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _f32c(t: torch.Tensor) -> torch.Tensor:
    assert t.is_cuda and t.dtype == torch.float32, "expected a CUDA fp32 tensor"
    return t.contiguous()


# ------------------------------------------------------------------------------------------------
# thin Python wrappers (tensor in / tensor out) used by the drop-in classes, the tests and bench.py
# ------------------------------------------------------------------------------------------------
_ws_tls = threading.local()


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Scratch for one C call, cached per (thread, device).  Per THREAD because ctypes releases the GIL: two host threads (e.g. one
    inside PrototypeMemory's lock running a search, one inside a classifier's device lock running the head) enqueue on the same
    stream, and a scratch buffer shared between them would be rewritten between two kernels of the other thread's call."""
    cache = getattr(_ws_tls, "ws", None)
    if cache is None:
        cache = _ws_tls.ws = {}
    key = (device.index if device.index is not None else torch.cuda.current_device())
    ws = cache.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes * 1.25) + 1024, dtype=torch.uint8, device=device)
        cache[key] = ws
    return ws


def knn_make_shadow(P: torch.Tensor) -> torch.Tensor:
    """fp16 (RNE) shadow of the prototype matrix for the tensor path's coarse pass"""
    L = load_library()
    P = _f32c(P)
    out = torch.empty(P.shape, dtype=torch.float16, device=P.device)
    check(L.ac_knn_make_shadow(P.data_ptr(), P.shape[0], P.shape[1], out.data_ptr(), stream_ptr()), "ac_knn_make_shadow")
    return out


def knn_l2_topk(Q: torch.Tensor, P: torch.Tensor, k: int, *, p_sqnorm: Optional[torch.Tensor] = None,
                p_half: Optional[torch.Tensor] = None, row_offset: int = 0, algo: int = AC_KNN_AUTO,
                stats: Optional[torch.Tensor] = None):
    """stats: optional CUDA int32[4] accumulator (see ac_knn_l2_topk): with it the call never synchronises and the CALLER must
    check stats[1] (buffer overflow -> redo those queries with AC_KNN_EXACT); without it the library does both itself."""
    L = load_library()
    Q = _f32c(Q)
    P = _f32c(P)
    B, D = Q.shape
    N = P.shape[0]
    assert P.shape[1] == D
    nbytes = c_size_t(0)
    check(L.ac_knn_workspace_bytes(B, N, D, k, algo, ctypes.byref(nbytes)), "ac_knn_workspace_bytes")
    ws = _workspace(nbytes.value, Q.device)
    out_d = torch.empty((B, k), dtype=torch.float32, device=Q.device)
    out_i = torch.empty((B, k), dtype=torch.int64, device=Q.device)
    check(L.ac_knn_l2_topk(Q.data_ptr(), P.data_ptr(), ptr(p_sqnorm), ptr(p_half), B, N, D, k, out_d.data_ptr(),
                           out_i.data_ptr(), row_offset, ws.data_ptr(), ws.numel(), algo, ptr(stats), stream_ptr()), "ac_knn_l2_topk")
    return out_d, out_i


def row_sqnorm(P: torch.Tensor) -> torch.Tensor:
    L = load_library()
    P = _f32c(P)
    out = torch.empty((P.shape[0],), dtype=torch.float32, device=P.device)
    check(L.ac_row_sqnorm(P.data_ptr(), P.shape[0], P.shape[1], out.data_ptr(), stream_ptr()), "ac_row_sqnorm")
    return out


def topk_merge(d: torch.Tensor, i: torch.Tensor):
    L = load_library()
    d = _f32c(d)
    i = i.contiguous()
    G, B, k = d.shape
    od = torch.empty((B, k), dtype=torch.float32, device=d.device)
    oi = torch.empty((B, k), dtype=torch.int64, device=d.device)
    check(L.ac_topk_merge(d.data_ptr(), i.data_ptr(), G, B, k, od.data_ptr(), oi.data_ptr(), stream_ptr()), "ac_topk_merge")
    return od, oi


def proto_scores(d: torch.Tensor, idx: Optional[torch.Tensor]) -> torch.Tensor:
    L = load_library()
    d = _f32c(d)
    B, k = d.shape
    out = torch.empty_like(d)
    check(L.ac_proto_scores(d.data_ptr(), ptr(idx.contiguous() if idx is not None else None), B, k, out.data_ptr(),
                            stream_ptr()), "ac_proto_scores")
    return out


def segment_mean(X: torch.Tensor, cls: torch.Tensor, C: int):
    L = load_library()
    X = _f32c(X)
    cls = cls.to(torch.int32).contiguous()
    n, D = X.shape
    mean = torch.zeros((C, D), dtype=torch.float32, device=X.device)
    cnt = torch.zeros((C,), dtype=torch.int32, device=X.device)
    check(L.ac_segment_mean(X.data_ptr(), cls.data_ptr(), n, D, C, mean.data_ptr(), cnt.data_ptr(), stream_ptr()),
          "ac_segment_mean")
    return mean, cnt


def memory_append_prune(rows, order, count, new_rows, new_index, cls_start, touched):
    """rows [n_slots, cap+1, D], order [n_slots, cap+1] int32, count [n_slots] int32 (updated in place) ->
    (src [n_touched, cap] int32, proto [n_touched, D] fp32): see ac_memory_append_prune"""
    L = load_library()
    n_slots, cap1, D = rows.shape
    nt = touched.numel()
    src = torch.empty((nt, cap1 - 1), dtype=torch.int32, device=rows.device)
    proto = torch.empty((nt, D), dtype=torch.float32, device=rows.device)
    ws = _workspace(nt * D * 8 + 256, rows.device)
    check(L.ac_memory_append_prune(rows.data_ptr(), order.data_ptr(), count.data_ptr(), cap1 - 1, D, _f32c(new_rows).data_ptr(),
                                   new_index.data_ptr(), cls_start.data_ptr(), touched.data_ptr(), nt, src.data_ptr(), proto.data_ptr(),
                                   ws.data_ptr(), ws.numel(), stream_ptr()), "ac_memory_append_prune")
    return src, proto


def head_params_struct(p: dict) -> HeadParams:
    """p: {'W0','b0','W1','b1','W2','b2'} CUDA fp32 contiguous tensors (nn.Linear layout)."""
    hp = HeadParams()
    hp.D = p["W0"].shape[1]
    hp.H0 = p["W0"].shape[0]
    hp.H1 = p["W1"].shape[0]
    hp.C = p["W2"].shape[0]
    for n in ("W0", "b0", "W1", "b1", "W2", "b2"):
        t = p[n]
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), n
        setattr(hp, n, t.data_ptr())
    return hp


def head_forward(X: torch.Tensor, p: dict, act: int = AC_ACT_LOGITS) -> torch.Tensor:
    L = load_library()
    X = _f32c(X)
    hp = head_params_struct(p)
    B = X.shape[0]
    out = torch.empty((B, hp.C), dtype=torch.float32, device=X.device)
    scratch = torch.empty((B * (hp.H0 + hp.H1),), dtype=torch.float32, device=X.device)
    check(L.ac_head_forward(X.data_ptr(), B, ctypes.byref(hp), act, out.data_ptr(), scratch.data_ptr(),
                            scratch.numel(), stream_ptr()), "ac_head_forward")
    return out


def head_train_step(X, targets, p, m, v, *, step, loss_kind=AC_LOSS_CE, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                    weight_decay=0.01, max_norm=1.0, dropout_p=0.1, masks=None, seed=0,
                    ewc=None, out_stats=None):
    """One optimizer step in place on p/m/v.  ewc = (fisher_dict, star_dict, lambda, C_old) or None.
    Returns the device tensor [task_loss, ewc_penalty, grad_norm]."""
    L = load_library()
    X = _f32c(X)
    B = X.shape[0]
    hp, hm, hv = head_params_struct(p), head_params_struct(m), head_params_struct(v)
    cfg = TrainCfg()
    cfg.lr, cfg.beta1, cfg.beta2, cfg.eps = lr, betas[0], betas[1], eps
    cfg.weight_decay, cfg.max_norm = weight_decay, max_norm
    cfg.step, cfg.loss_kind, cfg.dropout_p, cfg.seed = step, loss_kind, dropout_p, seed
    keep = []
    if masks is not None:
        m0, m1 = _f32c(masks[0]), _f32c(masks[1])
        keep += [m0, m1]
        cfg.mask0, cfg.mask1 = m0.data_ptr(), m1.data_ptr()
    if ewc is not None:
        fs, ss = head_params_struct(ewc[0]), head_params_struct(ewc[1])
        keep += [fs, ss]
        cfg.ewc_fisher, cfg.ewc_star = ctypes.pointer(fs), ctypes.pointer(ss)
        cfg.ewc_lambda, cfg.ewc_C_old = float(ewc[2]), int(ewc[3])
    nbytes = c_size_t(0)
    check(L.ac_head_train_workspace_bytes(B, 1, ctypes.byref(hp), ctypes.byref(nbytes)), "ac_head_train_workspace_bytes")
    ws = _workspace(nbytes.value, X.device)
    if out_stats is None:
        out_stats = torch.zeros((4,), dtype=torch.float32, device=X.device)
    targets = targets.contiguous()
    check(L.ac_head_train_step(X.data_ptr(), targets.data_ptr(), B, ctypes.byref(hp), ctypes.byref(hm),
                               ctypes.byref(hv), ctypes.byref(cfg), out_stats.data_ptr(), ws.data_ptr(), ws.numel(),
                               stream_ptr()), "ac_head_train_step")
    return out_stats


def head_train_epoch(X, targets, perm, p, m, v, *, first_step, batch, loss_kind=AC_LOSS_CE, lr=1e-3, betas=(0.9, 0.999),
                     eps=1e-8, weight_decay=0.01, max_norm=1.0, dropout_p=0.1, seed=0, ewc=None, loss_accum=None,
                     step_stats=None):
    """All optimizer steps of one epoch in ONE kernel launch (batches gathered on the device from `perm`).
    step_stats: optional CUDA fp32 [steps, 3] receiving (task loss, EWC penalty, grad norm) of every step.
    Returns (loss_accum tensor, steps)."""
    L = load_library()
    X = _f32c(X)
    n = X.shape[0]
    hp, hm, hv = head_params_struct(p), head_params_struct(m), head_params_struct(v)
    cfg = TrainCfg()
    cfg.lr, cfg.beta1, cfg.beta2, cfg.eps = lr, betas[0], betas[1], eps
    cfg.weight_decay, cfg.max_norm = weight_decay, max_norm
    cfg.step, cfg.loss_kind, cfg.dropout_p, cfg.seed = first_step, loss_kind, dropout_p, seed
    keep = []
    if ewc is not None:
        fs, ss = head_params_struct(ewc[0]), head_params_struct(ewc[1])
        keep += [fs, ss]
        cfg.ewc_fisher, cfg.ewc_star = ctypes.pointer(fs), ctypes.pointer(ss)
        cfg.ewc_lambda, cfg.ewc_C_old = float(ewc[2]), int(ewc[3])
    nbytes = c_size_t(0)
    steps = (n + batch - 1) // batch
    check(L.ac_head_train_workspace_bytes(batch, steps, ctypes.byref(hp), ctypes.byref(nbytes)), "ac_head_train_workspace_bytes")
    ws = _workspace(nbytes.value, X.device)
    if step_stats is not None:
        assert step_stats.is_cuda and step_stats.dtype == torch.float32 and step_stats.is_contiguous() and step_stats.numel() >= 3 * steps
    if loss_accum is None:
        loss_accum = torch.zeros((1,), dtype=torch.float32, device=X.device)
    targets = targets.contiguous()
    perm = perm.to(device=X.device, dtype=torch.int64).contiguous()
    check(L.ac_head_train_epoch(X.data_ptr(), targets.data_ptr(), perm.data_ptr(), n, batch, ctypes.byref(hp),
                                ctypes.byref(hm), ctypes.byref(hv), ctypes.byref(cfg), loss_accum.data_ptr(), ptr(step_stats),
                                ws.data_ptr(), ws.numel(), stream_ptr()), "ac_head_train_epoch")
    return loss_accum, steps


def head_phase_timing(enable: bool = True):
    """diagnostic: nanoseconds three observed CTAs of the training kernel (holders of a layer-0 / layer-1 / layer-2 block) spent per
    phase / grid barrier (13 counters) and inside the product routines (7 counters from index 14) since enabled: 3 lists of 24"""
    out = (ctypes.c_ulonglong * 72)()
    check(load_library().ac_head_phase_timing(1 if enable else 0, out), "ac_head_phase_timing")
    v = [int(x) for x in out]
    return [v[0:24], v[24:48], v[48:72]]


def head_train_plan(p, batch: int = 32):
    """diagnostic: {ctas, stages, moments_resident, smem_bytes} of the training kernel for this head"""
    hp = head_params_struct(p)
    out = (ctypes.c_int * 5)()
    check(load_library().ac_head_train_plan(batch, ctypes.byref(hp), out), "ac_head_train_plan")
    return dict(zip(("ctas", "stages", "moments_resident", "smem_bytes"), [int(x) for x in out][:4]))


def head_grad(X, targets, p, *, loss_kind=AC_LOSS_CE, grad_out=None, fisher=None, inv_n_batches=1.0):
    L = load_library()
    X = _f32c(X)
    B = X.shape[0]
    hp = head_params_struct(p)
    g = head_params_struct(grad_out) if grad_out is not None else None
    f = head_params_struct(fisher) if fisher is not None else None
    nbytes = c_size_t(0)
    check(L.ac_head_train_workspace_bytes(B, 1, ctypes.byref(hp), ctypes.byref(nbytes)), "ac_head_train_workspace_bytes")
    ws = _workspace(nbytes.value, X.device)
    loss = torch.zeros((1,), dtype=torch.float32, device=X.device)
    targets = targets.contiguous()
    check(L.ac_head_grad(X.data_ptr(), targets.data_ptr(), B, ctypes.byref(hp), loss_kind,
                         ctypes.byref(g) if g is not None else None, ctypes.byref(f) if f is not None else None,
                         float(inv_n_batches), loss.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr()), "ac_head_grad")
    return loss


def ewc_penalty(p, fisher, star, lam: float, batch_size: Optional[int], C_old: int = 0) -> torch.Tensor:
    L = load_library()
    hp, hf, hs = head_params_struct(p), head_params_struct(fisher), head_params_struct(star)
    out = torch.zeros((1,), dtype=torch.float32, device=p["W0"].device)
    inv = 1.0 / batch_size if batch_size else 1.0
    check(L.ac_ewc_penalty(ctypes.byref(hp), ctypes.byref(hf), ctypes.byref(hs), float(lam), float(inv), C_old,
                           out.data_ptr(), stream_ptr()), "ac_ewc_penalty")
    return out


def linear_tc(X, W, bias, residual=None, epi: int = 0, round_out: bool = False, out_half: bool = False) -> torch.Tensor:
    """X, W fp32 -> tf32 path; X, W fp16 -> fp16 path (the encoder's); Y fp32 unless out_half."""
    L = load_library()
    assert X.is_cuda and W.is_cuda and X.dtype == W.dtype and X.dtype in (torch.float32, torch.float16)
    X, W = X.contiguous(), W.contiguous()
    prec = AC_PREC_F16 if X.dtype == torch.float16 else AC_PREC_TF32
    M, K = X.shape
    N = W.shape[0]
    Y = torch.empty((M, N), dtype=torch.float16 if out_half else torch.float32, device=X.device)
    check(L.ac_linear_tc(X.data_ptr(), W.data_ptr(), ptr(bias), ptr(residual), Y.data_ptr(), M, N, K, epi,
                         1 if round_out else 0, prec, 1 if out_half else 0, stream_ptr()), "ac_linear_tc")
    return Y


def attention(qk: torch.Tensor, vT: torch.Tensor, mask: Optional[torch.Tensor], B: int, S: int, heads: int,
              window: int = 0) -> torch.Tensor:
    """The encoder's attention on caller buffers (see ac_attention): qk fp16 [rows >= B*S, 2H], vT fp16 [B*H, roundup(S, 8)],
    mask int32 [B, S] or None, window 0 = global -> ctx fp16 [B*S, H].  ctx starts as NaN, so a row the kernels never
    write cannot pass for a result."""
    L = load_library()
    H = 64 * heads
    assert qk.is_cuda and qk.dtype == torch.float16 and qk.is_contiguous() and qk.dim() == 2 and qk.shape[1] == 2 * H
    assert vT.is_cuda and vT.dtype == torch.float16 and vT.is_contiguous() and tuple(vT.shape) == (B * H, (S + 7) // 8 * 8)
    if mask is not None:
        mask = mask.to(device=qk.device, dtype=torch.int32).contiguous()
        assert tuple(mask.shape) == (B, S)
    ctx = torch.full((B * S, H), float("nan"), dtype=torch.float16, device=qk.device)
    check(L.ac_attention(qk.data_ptr(), qk.shape[0], vT.data_ptr(), ptr(mask), B, S, heads, window, ctx.data_ptr(),
                         stream_ptr()), "ac_attention")
    return ctx


def distilbert_to_bert_state_dict(sd: dict, c):
    """DistilBERT (HF models/distilbert/modeling_distilbert.py) is the BERT post-LN block without token-type embeddings:
    rename its parameters to the BERT names the encoder consumes and supply an all-zero single-row type table."""
    if getattr(c, "activation", "gelu") != "gelu" or getattr(c, "sinusoidal_pos_embds", False):
        raise AdaptiveB200Error("DistilBERT variant with non-GELU activation / sinusoidal positions is not implemented")
    out = {
        "embeddings.word_embeddings.weight": sd["embeddings.word_embeddings.weight"],
        "embeddings.position_embeddings.weight": sd["embeddings.position_embeddings.weight"],
        "embeddings.token_type_embeddings.weight": torch.zeros((1, c.dim), dtype=torch.float32),
        "embeddings.LayerNorm.weight": sd["embeddings.LayerNorm.weight"],
        "embeddings.LayerNorm.bias": sd["embeddings.LayerNorm.bias"],
    }
    ren = {"attention.q_lin": "attention.self.query", "attention.k_lin": "attention.self.key",
           "attention.v_lin": "attention.self.value", "attention.out_lin": "attention.output.dense",
           "sa_layer_norm": "attention.output.LayerNorm", "ffn.lin1": "intermediate.dense", "ffn.lin2": "output.dense",
           "output_layer_norm": "output.LayerNorm"}
    for l in range(c.n_layers):
        for src, dst in ren.items():
            for wb in ("weight", "bias"):
                out[f"encoder.layer.{l}.{dst}.{wb}"] = sd[f"transformer.layer.{l}.{src}.{wb}"]
    dims = dict(layers=c.n_layers, hidden=c.dim, heads=c.n_heads, intermediate=c.hidden_dim, vocab=c.vocab_size,
                max_pos=c.max_position_embeddings, type_vocab=1, ln_eps=1e-12, pad_idx=0)
    return out, dims


def modernbert_dims(c) -> dict:
    """HF ModernBertConfig -> the dimensions, per-layer key windows and rope thetas ac_encoder_create_modernbert takes.
    Pure (no device work), so that an unsupported checkpoint is refused before anything is allocated."""
    act = getattr(c, "hidden_activation", "gelu")
    if act != "gelu":
        raise AdaptiveB200Error(f"ModernBERT hidden_activation '{act}' is not implemented (exact-erf 'gelu' only)")
    H, nh, I = int(c.hidden_size), int(c.num_attention_heads), int(c.intermediate_size)
    if nh <= 0 or H % nh != 0 or H // nh != 64 or (getattr(c, "head_dim", None) or 64) != 64:
        raise AdaptiveB200Error(f"ModernBERT head_dim must be 64 (hidden_size={H}, num_attention_heads={nh})")
    if H % 128 != 0 or H > 1024:
        raise AdaptiveB200Error(f"ModernBERT hidden_size={H} must be a multiple of 128 and <= 1024")
    if I % 64 != 0:
        raise AdaptiveB200Error(f"ModernBERT intermediate_size={I} must be a multiple of 64")
    L = int(c.num_hidden_layers)
    types = list(getattr(c, "layer_types", None) or [])
    if len(types) != L:
        raise AdaptiveB200Error(f"ModernBERT layer_types has {len(types)} entries for {L} layers")
    rp = getattr(c, "rope_parameters", None) or {}
    windows, thetas = [], []
    for t in types:
        if t not in ("full_attention", "sliding_attention"):
            raise AdaptiveB200Error(f"ModernBERT layer type '{t}' is not implemented")
        p = rp.get(t) if isinstance(rp, dict) else None
        if not isinstance(p, dict) or "rope_theta" not in p:
            raise AdaptiveB200Error(f"ModernBERT rope_parameters carry no rope_theta for '{t}'")
        if p.get("rope_type", "default") != "default" or any(k not in ("rope_type", "rope_theta") for k in p):
            raise AdaptiveB200Error(f"ModernBERT rope scaling {p} is not implemented (rope_type 'default' only)")
        windows.append(int(c.sliding_window) if t == "sliding_attention" else 0)
        thetas.append(float(p["rope_theta"]))
    return dict(layers=L, hidden=H, heads=nh, intermediate=I, vocab=int(c.vocab_size), norm_eps=float(c.norm_eps),
                windows=windows, thetas=thetas)


class Encoder:
    """Owner of an ac_encoder handle built from an HF BERT/RoBERTa (or, through `modernbert`, ModernBERT) state_dict
    (CUDA fp32 tensors)."""

    def __init__(self, sd: dict, *, arch: str, layers: int, hidden: int, heads: int, intermediate: int, vocab: int,
                 max_pos: int, type_vocab: int, ln_eps: float, pad_idx: int = 0, max_tokens: int = 65536,
                 device="cuda", cls_only: bool = True):
        L = load_library()
        self._L = L
        self.hidden = hidden
        self.max_tokens = max_tokens
        dev = torch.device(device)
        keep = {}

        def g(name):
            t = sd[name].detach().to(device=dev, dtype=torch.float32).contiguous()
            keep[name] = t
            return t.data_ptr()

        def arr(fmt):
            a = (c_void_p * layers)(*[g(fmt.format(l)) for l in range(layers)])
            keep[fmt] = a
            return ctypes.cast(a, _PP)

        w = EncoderWeights()
        w.word_emb = g("embeddings.word_embeddings.weight")
        w.pos_emb = g("embeddings.position_embeddings.weight")
        w.type_emb = g("embeddings.token_type_embeddings.weight")
        w.emb_ln_w = g("embeddings.LayerNorm.weight")
        w.emb_ln_b = g("embeddings.LayerNorm.bias")
        p = "encoder.layer.{}."
        w.q_w, w.q_b = arr(p + "attention.self.query.weight"), arr(p + "attention.self.query.bias")
        w.k_w, w.k_b = arr(p + "attention.self.key.weight"), arr(p + "attention.self.key.bias")
        w.v_w, w.v_b = arr(p + "attention.self.value.weight"), arr(p + "attention.self.value.bias")
        w.ao_w, w.ao_b = arr(p + "attention.output.dense.weight"), arr(p + "attention.output.dense.bias")
        w.ao_ln_w, w.ao_ln_b = arr(p + "attention.output.LayerNorm.weight"), arr(p + "attention.output.LayerNorm.bias")
        w.ff1_w, w.ff1_b = arr(p + "intermediate.dense.weight"), arr(p + "intermediate.dense.bias")
        w.ff2_w, w.ff2_b = arr(p + "output.dense.weight"), arr(p + "output.dense.bias")
        w.out_ln_w, w.out_ln_b = arr(p + "output.LayerNorm.weight"), arr(p + "output.LayerNorm.bias")
        cfg = EncoderConfig(AC_ARCH_BERT if arch == "bert" else AC_ARCH_ROBERTA, layers, hidden, heads, intermediate,
                            vocab, max_pos, type_vocab, pad_idx, ln_eps, AC_PREC_F16, max_tokens, 1 if cls_only else 0)
        h = c_void_p()
        with torch.cuda.device(dev):
            check(L.ac_encoder_create(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(h)), "ac_encoder_create")
        self.handle = h
        del keep  # the handle holds its own packed copies

    @classmethod
    def modernbert(cls, sd: dict, dims: dict, *, max_tokens: int = 65536, device="cuda", cls_only: bool = True):
        """ac_encoder_create_modernbert over an HF ModernBertModel state_dict; dims = modernbert_dims(config)."""
        L = load_library()
        self = cls.__new__(cls)
        self._L = L
        self.hidden = dims["hidden"]
        self.max_tokens = max_tokens
        dev = torch.device(device)
        n = dims["layers"]
        keep = {}

        def g(name):
            t = sd.get(name)
            if t is None:
                return None
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            keep[name] = t
            return t.data_ptr()

        def arr(fmt, first=0):
            a = (c_void_p * n)(*[(g(fmt.format(l)) if l >= first else None) for l in range(n)])
            keep[fmt] = a
            return ctypes.cast(a, _PP)

        w = ModernBertEncoderWeights()
        w.tok_emb = g("embeddings.tok_embeddings.weight")
        w.emb_norm_w, w.emb_norm_b = g("embeddings.norm.weight"), g("embeddings.norm.bias")
        p = "layers.{}."
        w.attn_norm_w, w.attn_norm_b = arr(p + "attn_norm.weight", 1), arr(p + "attn_norm.bias", 1)
        w.Wqkv, w.Wqkv_b = arr(p + "attn.Wqkv.weight"), arr(p + "attn.Wqkv.bias")
        w.Wo, w.Wo_b = arr(p + "attn.Wo.weight"), arr(p + "attn.Wo.bias")
        w.mlp_norm_w, w.mlp_norm_b = arr(p + "mlp_norm.weight"), arr(p + "mlp_norm.bias")
        w.Wi, w.Wi_b = arr(p + "mlp.Wi.weight"), arr(p + "mlp.Wi.bias")
        w.mlp_Wo, w.mlp_Wo_b = arr(p + "mlp.Wo.weight"), arr(p + "mlp.Wo.bias")
        w.final_norm_w, w.final_norm_b = g("final_norm.weight"), g("final_norm.bias")
        win = (c_int * n)(*dims["windows"])
        th = (c_float * n)(*dims["thetas"])
        cfg = ModernBertEncoderConfig(n, dims["hidden"], dims["heads"], dims["intermediate"], dims["vocab"], dims["norm_eps"],
                                      AC_PREC_F16, max_tokens, 1 if cls_only else 0, win, th)
        h = c_void_p()
        with torch.cuda.device(dev):
            check(L.ac_encoder_create_modernbert(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(h)),
                  "ac_encoder_create_modernbert")
        self.handle = h
        del keep
        return self

    @classmethod
    def from_hf(cls, model, max_tokens: int = 65536, device="cuda", cls_only: bool = True):
        """Build from an in-memory HF BertModel / RobertaModel / DistilBertModel (post-LN blocks, head_dim 64) or
        ModernBertModel (pre-LN, RoPE, GeGLU, sliding-window layers)."""
        c = model.config
        mt = getattr(c, "model_type", "bert")
        if mt == "modernbert":
            dims = modernbert_dims(c)
            sd = {k: v for k, v in model.state_dict().items()}
            return cls.modernbert(sd, dims, max_tokens=max_tokens, device=device, cls_only=cls_only)
        sd = {k: v for k, v in model.state_dict().items()}
        if mt == "distilbert":
            sd, dims = distilbert_to_bert_state_dict(sd, c)
            return cls(sd, arch="bert", max_tokens=max_tokens, device=device, cls_only=cls_only, **dims)
        if mt not in ("bert", "roberta", "xlm-roberta"):
            raise AdaptiveB200Error(f"encoder architecture '{mt}' is not implemented in the B200 path yet")
        if getattr(c, "hidden_act", "gelu") != "gelu" or getattr(c, "position_embedding_type", "absolute") != "absolute":
            raise AdaptiveB200Error("only exact-erf GELU and absolute position embeddings are implemented")
        return cls(sd, arch="bert" if mt == "bert" else "roberta", layers=c.num_hidden_layers, hidden=c.hidden_size,
                   heads=c.num_attention_heads, intermediate=c.intermediate_size, vocab=c.vocab_size,
                   max_pos=c.max_position_embeddings, type_vocab=c.type_vocab_size, ln_eps=c.layer_norm_eps,
                   pad_idx=(c.pad_token_id if c.pad_token_id is not None else 0), max_tokens=max_tokens, device=device,
                   cls_only=cls_only)

    def forward_cls(self, ids: torch.Tensor, mask: Optional[torch.Tensor] = None,
                    type_ids: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        assert ids.is_cuda and ids.dtype == torch.int32 and ids.is_contiguous()
        B, S = ids.shape
        if out is None:
            out = torch.empty((B, self.hidden), dtype=torch.float32, device=ids.device)
        if mask is not None:
            mask = mask.to(torch.int32).contiguous()
        if type_ids is not None:
            type_ids = type_ids.to(torch.int32).contiguous()
        check(self._L.ac_encoder_forward_cls(self.handle, ids.data_ptr(), ptr(mask), ptr(type_ids), B, S,
                                             out.data_ptr(), stream_ptr()), "ac_encoder_forward_cls")
        return out

    def last_hidden(self, B: int, S: int) -> torch.Tensor:
        out = torch.empty((B * S, self.hidden), dtype=torch.float32, device="cuda")
        check(self._L.ac_encoder_last_hidden(self.handle, out.data_ptr(), out.numel(), stream_ptr()),
              "ac_encoder_last_hidden")
        return out

    def close(self):
        if getattr(self, "handle", None):
            self._L.ac_encoder_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def proto_class_scores(d, idx, row_class=None, n_classes: Optional[int] = None):
    """k <= 32: one thread per query; larger k (predict(): k = num_classes): one CTA per query, needs n_classes"""
    L = load_library()
    d = _f32c(d)
    idx = idx.contiguous()
    B, k = d.shape
    cls = torch.empty((B, k), dtype=torch.int32, device=d.device)
    sc = torch.empty((B, k), dtype=torch.float32, device=d.device)
    if k <= 32 and n_classes is None:
        check(L.ac_proto_class_scores(d.data_ptr(), idx.data_ptr(), ptr(row_class), B, k, cls.data_ptr(), sc.data_ptr(),
                                      stream_ptr()), "ac_proto_class_scores")
    else:
        assert n_classes is not None, "k > 32 needs the number of classes"
        check(L.ac_proto_class_scores_n(d.data_ptr(), idx.data_ptr(), ptr(row_class), B, k, int(n_classes), cls.data_ptr(),
                                        sc.data_ptr(), stream_ptr()), "ac_proto_class_scores_n")
    return cls, sc


def blend_dense(p_cls, p_score, head_probs, w_proto, w_head, kout: int):
    """predict() blend over all classes (classifier.py:446-480) -> (cls [B,kout] int32, score [B,kout])"""
    L = load_library()
    B, kp = p_cls.shape
    C = w_proto.numel()
    out_cls = torch.empty((B, kout), dtype=torch.int32, device=p_cls.device)
    out_sc = torch.empty((B, kout), dtype=torch.float32, device=p_cls.device)
    check(L.ac_blend_dense(p_cls.data_ptr(), _f32c(p_score).data_ptr(), kp, ptr(head_probs), B, C, _f32c(w_proto).data_ptr(),
                           ptr(w_head), kout, out_cls.data_ptr(), out_sc.data_ptr(), stream_ptr()), "ac_blend_dense")
    return out_cls, out_sc


def topk_desc(values: torch.Tensor, k: int):
    """-> (vals [B,k] descending, idx [B,k] int64); ties -> lower index."""
    L = load_library()
    values = _f32c(values)
    B, C = values.shape
    nbytes = c_size_t(0)
    check(L.ac_topk_desc_workspace_bytes(B, C, k, ctypes.byref(nbytes)), "ac_topk_desc_workspace_bytes")
    ws = _workspace(nbytes.value, values.device)
    neg = torch.empty((B, k), dtype=torch.float32, device=values.device)
    idx = torch.empty((B, k), dtype=torch.int64, device=values.device)
    check(L.ac_topk_desc(values.data_ptr(), B, C, k, neg.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws.numel(),
                         stream_ptr()), "ac_topk_desc")
    return -neg, idx


def blend_topk(p_cls, p_score, h_idx, h_val, k: int, w_proto: float = 0.7, w_head: float = 0.3):
    """h_val: head probabilities (descending) for h_idx, or None for prototype-only."""
    L = load_library()
    B = p_cls.shape[0]
    kh = 0 if h_idx is None else h_idx.shape[1]
    neg = (-h_val).contiguous() if h_val is not None else None
    out_cls = torch.empty((B, k), dtype=torch.int32, device=p_cls.device)
    out_sc = torch.empty((B, k), dtype=torch.float32, device=p_cls.device)
    check(L.ac_blend_topk(p_cls.data_ptr(), p_score.data_ptr(), ptr(h_idx), ptr(neg), B, k, kh, w_proto, w_head,
                          out_cls.data_ptr(), out_sc.data_ptr(), stream_ptr()), "ac_blend_topk")
    return out_cls, out_sc


def launch_count() -> int:
    return int(load_library().ac_launch_count())


def profile_enable(on: bool):
    check(load_library().ac_profile_enable(1 if on else 0), "ac_profile_enable")


def profile_read(cls: int):
    ms, fl, by = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
    n = ctypes.c_longlong(0)
    check(load_library().ac_profile_read(cls, ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(by), ctypes.byref(n)),
          "ac_profile_read")
    return {"ms": ms.value, "flops": fl.value, "bytes": by.value, "launches": n.value}


class _ExternalCudaBuffer:
    """__cuda_array_interface__ view of a device buffer owned by a C handle (fp32, row-major)"""

    def __init__(self, ptr_value: int, shape, device):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr_value), False), "version": 3,
                                         "strides": None}


class Pipeline:
    """ids -> E -> K -> class scores -> H -> blend, device or host (pinned) buffers at the boundary."""

    def __init__(self, enc: Encoder, P: torch.Tensor, max_B: int, S: int, k: int, *, head: Optional[dict] = None,
                 row_class: Optional[torch.Tensor] = None, p_sqnorm: Optional[torch.Tensor] = None,
                 p_half: Optional[torch.Tensor] = None, row_offset: int = 0, shards: int = 1):
        L = load_library()
        self._L = L
        self.enc, self.P, self.p_sqnorm, self.row_class, self.p_half = enc, _f32c(P), p_sqnorm, row_class, p_half
        self.head = head
        self.max_B, self.S, self.k = max_B, S, k
        hp = head_params_struct(head) if head is not None else None
        h = c_void_p()
        check(L.ac_pipeline_create(enc.handle, self.P.data_ptr(), ptr(p_sqnorm), ptr(p_half), ptr(row_class), self.P.shape[0],
                                   self.P.shape[1], ctypes.byref(hp) if hp is not None else None, max_B, S, k,
                                   row_offset, shards, ctypes.byref(h)), "ac_pipeline_create")
        self.handle = h
        self.shards = shards
        self.out_cls_host = torch.empty((max_B, k), dtype=torch.int32).pin_memory()
        self.out_score_host = torch.empty((max_B, k), dtype=torch.float32).pin_memory()
        self.out_cls = torch.empty((max_B, k), dtype=torch.int32, device=self.P.device)
        self.out_score = torch.empty((max_B, k), dtype=torch.float32, device=self.P.device)

    def predict_device(self, ids_dev: torch.Tensor, mask_dev: Optional[torch.Tensor] = None):
        B = ids_dev.shape[0]
        check(self._L.ac_pipeline_predict_device(self.handle, ids_dev.data_ptr(), ptr(mask_dev), B,
                                                 self.out_cls.data_ptr(), self.out_score.data_ptr(), stream_ptr()),
              "ac_pipeline_predict_device")
        return self.out_cls[:B], self.out_score[:B]

    def predict_host(self, ids_host: torch.Tensor):
        assert (not ids_host.is_cuda) and ids_host.dtype == torch.int32 and ids_host.is_contiguous()
        B = ids_host.shape[0]
        check(self._L.ac_pipeline_predict_host(self.handle, ids_host.data_ptr(), B, self.out_cls_host.data_ptr(),
                                               self.out_score_host.data_ptr(), stream_ptr()), "ac_pipeline_predict_host")
        return self.out_cls_host[:B], self.out_score_host[:B]

    # ---- phases of the row-sharded multi-GPU step (parallel.ShardedPipeline runs the collectives between them)
    def encode(self, ids_dev: torch.Tensor, mask_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
        """E (+ the head forked onto the side stream); returns a [B, D] view of the pipeline's embedding buffer"""
        B = ids_dev.shape[0]
        check(self._L.ac_pipeline_encode(self.handle, ids_dev.data_ptr(), ptr(mask_dev), B, stream_ptr()), "ac_pipeline_encode")
        if getattr(self, "_emb_view", None) is None:
            p = c_void_p()
            check(self._L.ac_pipeline_embeddings(self.handle, ctypes.byref(p)), "ac_pipeline_embeddings")
            D = self.P.shape[1]
            # wrap the handle-owned device buffer without copying (lifetime = the pipeline's)
            self._emb_store = _ExternalCudaBuffer(p.value, (self.max_B, D), self.P.device)
            self._emb_view = torch.as_tensor(self._emb_store, device=self.P.device)
        return self._emb_view[:B]

    def search_shard(self, q_all: torch.Tensor, G: int, B: int, packed: torch.Tensor) -> None:
        check(self._L.ac_pipeline_search_shard(self.handle, _f32c(q_all).data_ptr(), G, B, packed.data_ptr(), stream_ptr()),
              "ac_pipeline_search_shard")

    def finish_sharded(self, received: torch.Tensor, G: int, B: int):
        check(self._L.ac_pipeline_finish_sharded(self.handle, received.data_ptr(), G, B, self.out_cls.data_ptr(),
                                                 self.out_score.data_ptr(), stream_ptr()), "ac_pipeline_finish_sharded")
        return self.out_cls[:B], self.out_score[:B]

    def knn_stats(self, reset: bool = True) -> dict:
        """search statistics since the last reset (synchronises): queries that took the second tensor pass, queries whose
        candidate buffer overflowed (results not exact -> redo with AC_KNN_EXACT), max rows collected, searches"""
        out = (ctypes.c_int32 * 4)()
        check(self._L.ac_pipeline_knn_stats(self.handle, out, 1 if reset else 0, stream_ptr()), "ac_pipeline_knn_stats")
        return {"second_pass_queries": int(out[0]), "overflow_queries": int(out[1]), "max_collected": int(out[2]), "searches": int(out[3])}

    def debug_views(self, B: int):
        """(emb [B,D], knn_d [B,k], knn_i [B,k]) of the last call."""
        D = self.P.shape[1]
        emb = torch.empty((B, D), dtype=torch.float32, device=self.P.device)
        kd = torch.empty((B, self.k), dtype=torch.float32, device=self.P.device)
        ki = torch.empty((B, self.k), dtype=torch.int64, device=self.P.device)
        check(self._L.ac_pipeline_debug_copy(self.handle, B, emb.data_ptr(), kd.data_ptr(), ki.data_ptr(), stream_ptr()),
              "ac_pipeline_debug_copy")
        return emb, kd, ki

    def close(self):
        if getattr(self, "handle", None):
            self._L.ac_pipeline_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
