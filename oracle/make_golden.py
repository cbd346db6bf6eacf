"""Golden-vector generator (test infrastructure; runs ONLY in the dev container).

Imports the UNMODIFIED Python reference from /root/reference/src with oracle/shim/faiss.py standing in for
faiss-cpu (absent offline), drives it on seeded inputs and commits the resulting tensors as small fixtures
under tests/golden/.  /root/reference does not exist on the GPU box, so tests only read the fixtures.

    python oracle/make_golden.py            # rewrites tests/golden/*.npz

Fixtures
  golden_memory.npz      PrototypeMemory: adds -> prototypes, get_nearest_prototypes labels/scores
  golden_router.npz      the two real prototypes of scripts/adaptive_router/tensors.safetensors (6 KB,
                         inter-prototype d = 0.001965: near-tie stress) + reference search results
  golden_head.npz        AdaptiveHead forward / EWC loss values of the reference on seeded inputs
  golden_classifier.npz  digest + vocab of the tiny seeded BERT checkpoint (oracle/tiny_bert.py rebuilds it), reference
                         _get_embeddings / add_examples / predict / predict_batch outputs and the reference-trained head
  golden_training.npz    the reference's two training loops (_train_adaptive_head, _train_new_classes + EWC/Fisher)
                         run UNMODIFIED with recorders hooked onto torch/numpy entry points: the dataset of every
                         training call, every batch index list the DataLoader yielded, np.random.choice draws,
                         the Fisher batches' sampled labels, per-step loss and pre-clip grad norm, head state before
                         and after.  nn.Dropout is patched to identity for this fixture only (CPU mt19937 masks
                         cannot be reproduced on a GPU); everything else is the stock code path.
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "shim"))
sys.path.insert(0, "/root/reference/src")
sys.path.insert(0, ROOT)
from oracle import tiny_bert  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def unit(x):
    return x / x.norm(dim=-1, keepdim=True)


def gen_memory():
    from adaptive_classifier.memory import PrototypeMemory
    from adaptive_classifier.models import Example, ModelConfig
    g = torch.Generator().manual_seed(11)
    D = 64
    labels = ["alpha", "beta", "gamma"]
    centres = unit(torch.randn(3, D, generator=g))
    embs, labs = [], []
    for i in range(60):
        c = i % 3
        embs.append(unit(centres[c] + 0.3 * torch.randn(D, generator=g) / D ** 0.5 * 4))
        labs.append(labels[c])
    mem = PrototypeMemory(D, config=ModelConfig({"prototype_update_frequency": 25, "max_examples_per_class": 15}))
    for e, l in zip(embs, labs):
        mem.add_example(Example(f"t{len(l)}", l, e), l)
    mem._rebuild_index()
    queries = unit(torch.randn(8, D, generator=g) * 0.2 + centres[torch.arange(8) % 3])
    res_labels, res_scores = [], []
    for q in queries:
        r = mem.get_nearest_prototypes(q, k=3)
        res_labels.append([labels.index(l) for l, _ in r])
        res_scores.append([s for _, s in r])
    r2 = mem.get_nearest_prototypes(queries[0], k=2)
    np.savez_compressed(
        os.path.join(OUT, "golden_memory.npz"),
        embeddings=torch.stack(embs).numpy(), label_ids=np.array([labels.index(l) for l in labs]),
        labels=np.array(labels), queries=queries.numpy(),
        prototypes=torch.stack([mem.prototypes[l] for l in sorted(mem.prototypes)]).numpy(),
        kept=np.array([len(mem.examples[l]) for l in labels]),
        res_labels=np.array(res_labels), res_scores=np.array(res_scores, dtype=np.float64),
        res_k2_labels=np.array([labels.index(l) for l, _ in r2]), res_k2_scores=np.array([s for _, s in r2]),
        updates_since_rebuild=np.array(mem.updates_since_rebuild))
    print("golden_memory ok")


def gen_router():
    import faiss
    from safetensors.torch import load_file
    t = load_file("/root/reference/scripts/adaptive_router/tensors.safetensors")
    P = torch.stack([t["prototype_HIGH"], t["prototype_LOW"]]).float()
    g = torch.Generator().manual_seed(5)
    Q = unit(P[torch.arange(12) % 2] + 0.02 * torch.randn(12, P.shape[1], generator=g))
    idx = faiss.IndexFlatL2(P.shape[1])
    idx.add(P.numpy())
    d, i = idx.search(Q.numpy(), 2)
    np.savez_compressed(os.path.join(OUT, "golden_router.npz"), P=P.numpy(), Q=Q.numpy(), d=d, i=i)
    print("golden_router ok; inter-prototype d =", float(((P[0] - P[1]) ** 2).sum()))


def gen_head():
    from adaptive_classifier.models import AdaptiveHead
    from adaptive_classifier.ewc import EWC
    D, C = 64, 5
    head = AdaptiveHead(D, C, hidden_dims=[D, D // 2])
    head.eval()
    g = torch.Generator().manual_seed(21)
    X = unit(torch.randn(16, D, generator=g))
    with torch.no_grad():
        logits = head(X)
    sd = {k: v.numpy().copy() for k, v in head.state_dict().items()}
    # EWC identities of tests/test_ewc.py:128-153 on the reference: loss == 0 at theta*, > 0 after +0.1
    ds = torch.utils.data.TensorDataset(X, torch.randint(0, C, (16,), generator=g))
    torch.manual_seed(0)
    ewc = EWC(head, ds, device="cpu", ewc_lambda=100.0)
    loss0 = float(ewc.ewc_loss())
    with torch.no_grad():
        for p in head.parameters():
            p.add_(0.1)
    loss1 = float(ewc.ewc_loss())
    loss1_b32 = float(ewc.ewc_loss(batch_size=32))
    fisher = {("fisher_" + k): v.numpy().copy() for k, v in ewc.fisher_info.items()}
    np.savez_compressed(os.path.join(OUT, "golden_head.npz"), X=X.numpy(), logits=logits.numpy().copy(),
                        ewc_loss0=loss0, ewc_loss1=loss1, ewc_loss1_b32=loss1_b32, **sd, **fisher)
    print("golden_head ok", loss0, loss1, loss1_b32)


def gen_classifier():
    from adaptive_classifier import AdaptiveClassifier
    tmp, words, vocab, model, cfg = _tiny_checkpoint()

    rng = np.random.default_rng(7)
    class_words = {"sports": words[0:40], "finance": words[40:80], "cooking": words[80:120]}

    def sentence(label, n):
        own = rng.choice(class_words[label], size=n, replace=True)
        noise = rng.choice(words[120:], size=max(1, n // 4), replace=True)
        toks = list(own) + list(noise)
        rng.shuffle(toks)
        return " ".join(toks)

    texts, labels = [], []
    for label in ["sports", "finance", "cooking"]:
        for _ in range(12):
            texts.append(sentence(label, int(rng.integers(4, 14))))
            labels.append(label)
    test_texts = [sentence(l, 9) for l in ["sports", "finance", "cooking", "finance", "sports", "cooking"]]

    torch.manual_seed(0)
    np.random.seed(0)
    clf = AdaptiveClassifier(tmp, device="cpu", use_onnx=False)
    clf.add_examples(texts[:24], labels[:24])           # sports + finance -> _train_adaptive_head
    clf.add_examples(texts[24:], labels[24:])           # new class cooking -> _train_new_classes (+EWC)
    emb_train = torch.stack(clf._get_embeddings(texts)).numpy()
    emb_test = torch.stack(clf._get_embeddings(test_texts)).numpy()
    enc = clf.tokenizer(texts + test_texts, max_length=512, truncation=True, padding=True, return_tensors="pt")
    label_names = [clf.id_to_label[i] for i in range(len(clf.id_to_label))]
    pred = [clf.predict(t, k=3) for t in test_texts]
    pred_k1 = [clf.predict(t, k=1) for t in test_texts]
    pred_b = clf.predict_batch(test_texts, k=2)
    train_top1 = [p[0][0] for p in clf.predict_batch(texts, k=1)]     # end metric of the reference's own training

    def pack(preds, k):
        L = np.full((len(preds), k), -1, dtype=np.int64)
        S = np.zeros((len(preds), k), dtype=np.float64)
        for i, p in enumerate(preds):
            for j, (l, s) in enumerate(p):
                L[i, j] = label_names.index(l)
                S[i, j] = s
        return L, S

    pl, ps = pack(pred, 3)
    p1l, p1s = pack(pred_k1, 1)
    pbl, pbs = pack(pred_b, 2)
    head_sd = {("head_" + k): v.detach().numpy() for k, v in clf.adaptive_head.state_dict().items()}
    protos = np.stack([clf.memory.prototypes[l].numpy() for l in sorted(clf.memory.prototypes)])
    np.savez_compressed(
        os.path.join(OUT, "golden_classifier.npz"),
        vocab=np.array(vocab), texts=np.array(texts), labels=np.array(labels), test_texts=np.array(test_texts),
        label_names=np.array(label_names), input_ids=enc["input_ids"].numpy(), attention_mask=enc["attention_mask"].numpy(),
        emb_train=emb_train, emb_test=emb_test, prototypes=protos, proto_labels=np.array(sorted(clf.memory.prototypes)),
        training_history=json.dumps(clf.training_history), train_steps=clf.train_steps,
        pred_labels=pl, pred_scores=ps, pred_k1_labels=p1l, pred_k1_scores=p1s, predb_labels=pbl, predb_scores=pbs,
        train_top1=np.array([label_names.index(l) for l in train_top1]),
        bert_config=json.dumps(cfg.to_dict()), bert_sha256=tiny_bert.digest(model.state_dict()), **head_sd)
    print("golden_classifier ok; labels", label_names, "pred[0]", pred[0])


def _tiny_checkpoint():
    """the seeded tiny BERT of oracle/tiny_bert.py + its vocab on disk"""
    model, cfg = tiny_bert.build()
    tmp = tiny_bert.save_checkpoint(model, tempfile.mkdtemp(prefix="golden_ckpt_"))
    return tmp, tiny_bert.WORDS, tiny_bert.VOCAB, model, cfg


class _Recorder:
    """Hooks (installed around the unmodified reference, removed afterwards) on the library entry points its training
    loops call: TensorDataset() (the dataset of a loop), BatchSampler.__iter__ (index lists), np.random.choice,
    torch.multinomial (Fisher labels), CrossEntropyLoss / BCELoss forward (per-step loss), clip_grad_norm_ (grad norm)."""

    def __init__(self):
        self.events = []

    def __enter__(self):
        import torch.utils.data as tud
        import torch.nn as nn
        self._saved = []
        rec = self

        def patch(obj, name, make):
            orig = getattr(obj, name)
            self._saved.append((obj, name, orig))
            setattr(obj, name, make(orig))

        def mk_ds(orig):
            def init(self_, *tensors):
                rec.events.append(("dataset", [t.detach().cpu().clone() for t in tensors]))
                return orig(self_, *tensors)
            return init
        patch(tud.TensorDataset, "__init__", mk_ds)

        def mk_bs(orig):
            def it(self_):
                for b in orig(self_):
                    rec.events.append(("batch", list(b)))
                    yield b
                rec.events.append(("epoch_end", None))
            return it
        patch(tud.sampler.BatchSampler, "__iter__", mk_bs)

        def mk_choice(orig):
            def choice(a, size=None, replace=True, p=None):
                r = orig(a, size=size, replace=replace, p=p)
                rec.events.append(("choice", (int(a), int(size), bool(replace), np.asarray(r).copy())))
                return r
            return choice
        patch(np.random, "choice", mk_choice)

        def mk_multi(orig):
            def multinomial(probs, n, *a, **k):
                r = orig(probs, n, *a, **k)
                rec.events.append(("multinomial", r.detach().cpu().clone()))
                return r
            return multinomial
        patch(torch, "multinomial", mk_multi)

        def mk_loss(kind):
            def mk(orig):
                def fwd(self_, inp, tgt):
                    r = orig(self_, inp, tgt)
                    rec.events.append(("loss", (kind, float(r.detach()))))
                    return r
                return fwd
            return mk
        patch(nn.CrossEntropyLoss, "forward", mk_loss("ce"))
        patch(nn.BCELoss, "forward", mk_loss("bce"))

        def mk_clip(orig):
            def clip(params, max_norm, *a, **k):
                r = orig(params, max_norm, *a, **k)
                rec.events.append(("gnorm", float(r)))
                return r
            return clip
        patch(torch.nn.utils, "clip_grad_norm_", mk_clip)
        patch(nn.Dropout, "forward", lambda orig: (lambda self_, x: x))       # identity: see the module docstring
        return self

    def __exit__(self, *exc):
        for obj, name, orig in reversed(self._saved):
            setattr(obj, name, orig)


def _split_calls(events):
    """event stream -> one record per DataLoader-driven loop: dataset tensors, list of epochs (each a list of batches),
    per-step losses / grad norms, np.random.choice draws and multinomial draws that preceded it"""
    loops, cur, pending_choice, pending_multi = [], None, [], []
    last_ds = None
    for kind, val in events:
        if kind == "dataset":
            last_ds = val
        elif kind == "choice":
            pending_choice.append(val)
        elif kind == "batch":
            if cur is None or cur["closed"]:
                cur = {"dataset": last_ds, "epochs": [[]], "loss": [], "gnorm": [], "multinomial": [], "closed": False,
                       "choice": pending_choice}
                pending_choice = []
                loops.append(cur)
            cur["epochs"][-1].append(val)
        elif kind == "epoch_end":
            cur["epochs"].append([])
        elif kind == "loss":
            cur["loss"].append(val)
        elif kind == "gnorm":
            cur["gnorm"].append(val)
        elif kind == "multinomial":
            cur["multinomial"].append(val)
        elif kind == "loop_end":
            cur["closed"] = True
    for l in loops:
        l["epochs"] = [e for e in l["epochs"] if e]
    return loops


def gen_training():
    """SURVEY 8(c).3 / VERDICT r1 #5: loop-level goldens of H3 (classifier.py:1428-1522), H4 (:202-367), H5's Fisher
    (ewc.py:39-94) and the multilabel BCE loop (multilabel.py:309-413), recorded from the unmodified reference."""
    from adaptive_classifier import AdaptiveClassifier, MultiLabelAdaptiveClassifier
    tmp, words, vocab, _model, _cfg = _tiny_checkpoint()
    rng = np.random.default_rng(17)
    class_words = {"sports": words[0:40], "finance": words[40:80], "cooking": words[80:120]}

    def sentence(labels, n):
        pool = sum((class_words[l] for l in labels), [])
        toks = list(rng.choice(pool, size=n, replace=True)) + list(rng.choice(words[120:], size=max(1, n // 4), replace=True))
        rng.shuffle(toks)
        return " ".join(toks)

    names = ["sports", "finance", "cooking"]
    texts = {l: [sentence([l], int(rng.integers(4, 14))) for _ in range(30)] for l in names}
    out = {}

    def state(head):
        return {k: v.detach().cpu().numpy().copy() for k, v in head.state_dict().items()}

    def dump(prefix, loop, before, after):
        out[prefix + "X"] = loop["dataset"][0].numpy()
        out[prefix + "Y"] = loop["dataset"][1].numpy()
        sizes = [len(b) for e in loop["epochs"] for b in e]
        out[prefix + "batches"] = np.array([i for e in loop["epochs"] for b in e for i in b], dtype=np.int64)
        out[prefix + "batch_sizes"] = np.array(sizes, dtype=np.int64)
        out[prefix + "steps_per_epoch"] = np.array([len(e) for e in loop["epochs"]], dtype=np.int64)
        out[prefix + "loss"] = np.array([v for _, v in loop["loss"]], dtype=np.float64)
        out[prefix + "gnorm"] = np.array(loop["gnorm"], dtype=np.float64)
        for k, v in before.items():
            out[prefix + "before_" + k] = v
        for k, v in after.items():
            out[prefix + "after_" + k] = v

    # ---- single-label: call 1 -> _train_adaptive_head (H3); call 2 adds a class -> _train_new_classes (H4) with EWC/Fisher
    torch.manual_seed(0)
    np.random.seed(0)
    clf = AdaptiveClassifier(tmp, device="cpu", use_onnx=False)
    t1 = texts["sports"] + texts["finance"]
    l1 = ["sports"] * 30 + ["finance"] * 30
    with _Recorder() as rec:
        orig_init = clf._initialize_adaptive_head
        holder = {}

        def init_and_snapshot():
            orig_init()
            holder["before"] = state(clf.adaptive_head)
        clf._initialize_adaptive_head = init_and_snapshot
        clf.add_examples(t1, l1)
    loops = _split_calls(rec.events)
    assert len(loops) == 1, len(loops)
    dump("h3_", loops[0], holder["before"], state(clf.adaptive_head))
    out["h3_texts"] = np.array(t1)
    out["h3_labels"] = np.array(l1)

    with _Recorder() as rec:
        orig_upd = clf.adaptive_head.update_num_classes.__func__
        head_cls = type(clf.adaptive_head)

        def upd(self_, n):
            orig_upd(self_, n)
            holder["before4"] = state(self_)
        head_cls.update_num_classes = upd
        try:
            clf.add_examples(texts["cooking"], ["cooking"] * 30)
        finally:
            head_cls.update_num_classes = orig_upd
    ev = rec.events
    # the Fisher loop (global-RNG DataLoader) runs first, then the training loop: mark the boundary
    marked, seen_multi = [], False
    for e in ev:
        marked.append(e)
        if e[0] == "multinomial":
            seen_multi = True
        if e[0] == "epoch_end" and seen_multi:       # the Fisher pass is a single epoch
            marked.append(("loop_end", None))
            seen_multi = False
    # datasets: [old_dataset (EWC), dataset (training)] in construction order -- classifier.py:273 builds the training dataset
    # BEFORE the EWC one, so resolve by shapes below instead of by order
    loops = _split_calls(marked)
    fisher_loop = [l for l in loops if l["multinomial"]]
    train_loop = [l for l in loops if not l["multinomial"]]
    assert len(fisher_loop) == 1 and len(train_loop) == 1, (len(fisher_loop), len(train_loop))
    datasets = [v for k, v in ev if k == "dataset"]
    n_train = sum(len(b) for b in train_loop[0]["epochs"][0])
    train_loop[0]["dataset"] = [d for d in datasets if d[0].shape[0] == n_train][0]
    n_f = sum(len(b) for b in fisher_loop[0]["epochs"][0])
    fisher_loop[0]["dataset"] = [d for d in datasets if d[0].shape[0] == n_f and d[0].shape[0] != n_train][0]
    dump("h4_", train_loop[0], holder["before4"], state(clf.adaptive_head))
    ch = train_loop[0]["choice"] + fisher_loop[0]["choice"]
    out["h4_choice_args"] = np.array([[a, s, int(r)] for a, s, r, _ in ch], dtype=np.int64)
    out["h4_choice_idx"] = np.concatenate([c[3].reshape(-1) for c in ch]).astype(np.int64)
    out["h4_fisher_X"] = fisher_loop[0]["dataset"][0].numpy()
    out["h4_fisher_Y"] = fisher_loop[0]["dataset"][1].numpy()
    out["h4_fisher_batches"] = np.array([i for b in fisher_loop[0]["epochs"][0] for i in b], dtype=np.int64)
    out["h4_fisher_batch_sizes"] = np.array([len(b) for b in fisher_loop[0]["epochs"][0]], dtype=np.int64)
    out["h4_fisher_sampled"] = torch.cat([m.reshape(-1) for m in fisher_loop[0]["multinomial"]]).numpy()
    out["h4_new_texts"] = np.array(texts["cooking"])
    out["h4_memory_order"] = np.array(list(clf.memory.examples.keys()))
    out["h4_label_names"] = np.array([clf.id_to_label[i] for i in range(len(clf.id_to_label))])
    emb_all = torch.stack(clf._get_embeddings(t1 + texts["cooking"])).numpy()
    out["h4_emb_all"] = emb_all
    out["h4_train_top1"] = np.array([out["h4_label_names"].tolist().index(p[0][0])
                                     for p in clf.predict_batch(t1 + texts["cooking"], k=1)])

    # ---- multilabel BCE loop (multilabel.py:309-413)
    torch.manual_seed(0)
    np.random.seed(0)
    ml = MultiLabelAdaptiveClassifier(tmp, device="cpu")
    ml_texts, ml_labels = [], []
    combos = [["sports"], ["finance"], ["cooking"], ["sports", "finance"], ["finance", "cooking"], ["sports", "cooking"]]
    for i in range(48):
        labs = combos[i % len(combos)]
        ml_texts.append(sentence(labs, int(rng.integers(6, 14))))
        ml_labels.append(labs)
    with _Recorder() as rec:
        orig_init = ml._initialize_adaptive_head

        def init_and_snapshot_ml():
            orig_init()
            holder["before_ml"] = state(ml.adaptive_head)
        ml._initialize_adaptive_head = init_and_snapshot_ml
        ml.add_examples(ml_texts, ml_labels)
    loops = _split_calls(rec.events)
    assert len(loops) == 1, len(loops)
    dump("ml_", loops[0], holder["before_ml"], state(ml.adaptive_head))
    out["ml_texts"] = np.array(ml_texts)
    out["ml_labels"] = np.array(["|".join(l) for l in ml_labels])
    out["ml_label_names"] = np.array([ml.id_to_label[i] for i in range(len(ml.id_to_label))])
    test = [sentence(c, 10) for c in combos]
    enc = ml.tokenizer(ml_texts + test, max_length=512, truncation=True, padding=True, return_tensors="pt")
    out["ml_input_ids"] = enc["input_ids"].numpy()
    out["ml_attention_mask"] = enc["attention_mask"].numpy()
    out["ml_test_texts"] = np.array(test)
    preds = [ml.predict_multilabel(t) for t in test]
    out["ml_pred"] = np.array([json.dumps(p) for p in preds])
    out["ml_thresholds"] = np.array(json.dumps(ml.label_thresholds))
    out["bert_config"] = np.array(json.dumps(clf.model.config.to_dict()))
    out["vocab"] = np.array(vocab)
    out["bert_sha256"] = np.array(tiny_bert.digest(clf.model.state_dict()))
    np.savez_compressed(os.path.join(OUT, "golden_training.npz"), **out)
    print("golden_training ok: h3 steps", len(out["h3_loss"]), "epochs", len(out["h3_steps_per_epoch"]),
          "| h4 steps", len(out["h4_loss"]), "epochs", len(out["h4_steps_per_epoch"]), "rows", out["h4_X"].shape,
          "| fisher batches", len(out["h4_fisher_batch_sizes"]), "| ml steps", len(out["ml_loss"]), "preds", preds[:2])


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    only = sys.argv[1:]
    for name, fn in [("memory", gen_memory), ("router", gen_router), ("head", gen_head), ("classifier", gen_classifier),
                     ("training", gen_training)]:
        if not only or name in only:
            fn()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
