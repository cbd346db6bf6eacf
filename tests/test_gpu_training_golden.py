"""GPU parity of the two training loops (SURVEY.md 8(a) H3 / H4, 8(c).3) against the reference's OWN run.

tests/golden/golden_training.npz was recorded by oracle/make_golden.py::gen_training from the unmodified reference
(`_train_adaptive_head` classifier.py:1428-1522, `_train_new_classes` :202-367, the multilabel BCE loop multilabel.py:309-413)
with nn.Dropout as identity: the dataset of every loop, every batch index list its DataLoader yielded, the np.random.choice
draws, per-step loss and pre-clip grad norm, the head before and after.  Here the product's loop (`_run_epochs` ->
ac_head_train_epoch, through the C ABI) is replayed with dropout 0 on the same dataset and initial head and must reproduce the
batch order, the epoch count (early stopping / ReduceLROnPlateau), every step's loss to 1e-5 and the final weights to 1e-4."""
import json
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
NAMES = {"W0": "model.0.weight", "b0": "model.0.bias", "W1": "model.3.weight", "b1": "model.3.bias",
         "W2": "model.6.weight", "b2": "model.6.bias"}


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLD, "golden_training.npz"))


@pytest.fixture(scope="module")
def acb(cabi):
    import adaptive_classifier_b200 as m
    return m


def _batches(g, prefix):
    sizes, flat = g[prefix + "batch_sizes"].tolist(), g[prefix + "batches"].tolist()
    out, c = [], 0
    for s in sizes:
        out.append(flat[c:c + s])
        c += s
    return out


def _bare(acb, head, loss_kind):
    """the training half of AdaptiveClassifier without an encoder: `_run_epochs` only touches adaptive_head / _loss_kind"""
    clf = acb.AdaptiveClassifier.__new__(acb.AdaptiveClassifier)
    clf.adaptive_head = head
    clf._loss_kind = loss_kind
    clf._dropout_p = 0.0
    clf.device = "cuda"
    return clf


@pytest.mark.parametrize("prefix,epochs,sched,kind", [("h3_", 10, True, "ce"), ("h4_", 15, False, "ce"), ("ml_", 10, False, "bce")])
def test_product_loop_replays_the_reference_run(acb, cabi, g, prefix, epochs, sched, kind):
    X = torch.from_numpy(g[prefix + "X"]).cuda()
    Y = torch.from_numpy(g[prefix + "Y"]).cuda()
    D, C = X.shape[1], g[prefix + "before_model.6.weight"].shape[0]
    cls = acb.MultiLabelAdaptiveHead if kind == "bce" else acb.AdaptiveHead
    head = cls(D, C, hidden_dims=[D, D // 2])
    head.load_state_dict({v: torch.from_numpy(g[prefix + "before_" + v]) for v in NAMES.values()})
    head = head.cuda()
    bare = _bare(acb, head, cabi.AC_LOSS_BCE if kind == "bce" else cabi.AC_LOSS_CE)
    bs = min(32, X.shape[0])
    bare._run_epochs(X, Y, epochs=epochs, batch_size=bs, use_scheduler=sched)
    tr = bare.last_training_trace
    assert tr["steps_per_epoch"] == g[prefix + "steps_per_epoch"].tolist()           # same early-stopping decision
    assert np.abs(np.array(tr["loss"]) - g[prefix + "loss"]).max() < 1e-5             # every optimizer step's loss
    assert np.abs(np.array(tr["gnorm"]) - g[prefix + "gnorm"]).max() < 1e-4
    sd = head.state_dict()
    for v in NAMES.values():
        assert (sd[v].cpu() - torch.from_numpy(g[prefix + "after_" + v])).abs().max().item() < 1e-4, v


def test_product_batch_order_is_the_dataloaders(g):
    """CPU-only logic, kept next to its GPU consumer: the index lists the reference's DataLoader yielded, epoch by epoch"""
    from adaptive_classifier_b200.classifier import dataloader_epoch_permutation
    for prefix in ("h3_", "h4_", "ml_"):
        n = g[prefix + "X"].shape[0]
        bs = min(32, n)
        gen = torch.Generator().manual_seed(42)
        mine = []
        for _ in g[prefix + "steps_per_epoch"]:
            perm = dataloader_epoch_permutation(gen, n).tolist()
            mine += [perm[i:i + bs] for i in range(0, n, bs)]
        assert mine == _batches(g, prefix)


@pytest.fixture(scope="module")
def ckpt_dir(g):
    from oracle import tiny_bert
    assert g["vocab"].tolist() == tiny_bert.VOCAB
    m, _ = tiny_bert.model(g["bert_sha256"])
    return tiny_bert.save_checkpoint(m, tempfile.mkdtemp(prefix="golden_train_ckpt_"))


def test_add_examples_end_to_end_follows_the_reference_run(acb, g, ckpt_dir, monkeypatch):
    """The whole add_examples path (encoder -> memory -> H3, then a new class -> resampling -> Fisher -> H4) on the texts of the
    reference run with dropout 0: the np.random.choice draws are identical, the loops stop after the same number of epochs,
    step losses follow the reference's within the encoder's fp16-operand tolerance, and the end metric (top-1 of every
    training text) is the reference's."""
    draws = []
    orig = np.random.choice

    def rec(a, size=None, replace=True, p=None):
        r = orig(a, size=size, replace=replace, p=p)
        draws.append((int(a), int(size), int(bool(replace)), np.asarray(r).copy()))
        return r
    monkeypatch.setattr(np.random, "choice", rec)
    monkeypatch.setattr(acb.AdaptiveClassifier, "_dropout_p", 0.0)
    torch.manual_seed(0)
    np.random.seed(0)
    clf = acb.AdaptiveClassifier(ckpt_dir, device="cuda")
    t1, l1 = g["h3_texts"].tolist(), g["h3_labels"].tolist()
    clf.add_examples(t1, l1)
    tr = clf.last_training_trace
    assert tr["steps_per_epoch"] == g["h3_steps_per_epoch"].tolist()
    assert np.abs(np.array(tr["loss"]) - g["h3_loss"]).max() < 2e-3
    new_texts = g["h4_new_texts"].tolist()
    n_new = len(new_texts)
    assert n_new == 30 and g["h4_emb_all"].shape[0] == len(t1) + n_new
    clf.add_examples(new_texts, ["cooking"] * n_new)
    tr = clf.last_training_trace
    assert [d[:3] for d in draws] == [tuple(r) for r in g["h4_choice_args"].tolist()]
    assert np.array_equal(np.concatenate([d[3].reshape(-1) for d in draws]), g["h4_choice_idx"])
    assert tr["steps_per_epoch"] == g["h4_steps_per_epoch"].tolist()
    assert np.abs(np.array(tr["loss"]) - g["h4_loss"]).max() < 5e-3
    names = g["h4_label_names"].tolist()
    assert [clf.id_to_label[i] for i in range(3)] == names
    emb = torch.stack(clf._get_embeddings(t1 + new_texts)).numpy()
    assert np.linalg.norm(emb - g["h4_emb_all"], axis=1).max() < 1e-3
    top1 = [names.index(p[0][0]) for p in clf.predict_batch(t1 + new_texts, k=1)]
    assert np.mean(np.array(top1) == g["h4_train_top1"]) >= 0.97          # a fp16-operand near-tie may flip one of 90


def test_multilabel_predictions_follow_the_reference_run(acb, g, ckpt_dir, monkeypatch):
    """multilabel.py:132-229 (predict_multilabel) after the BCE loop of multilabel.py:309-413, dropout 0"""
    monkeypatch.setattr(acb.AdaptiveClassifier, "_dropout_p", 0.0)
    torch.manual_seed(0)
    np.random.seed(0)
    ml = acb.MultiLabelAdaptiveClassifier(ckpt_dir, device="cuda")
    texts = g["ml_texts"].tolist()
    labels = [s.split("|") for s in g["ml_labels"].tolist()]
    # the reference's multilabel head is default-initialised from the (unseeded) global RNG state of that run (multilabel.py:27-36):
    # start from the recorded initial weights
    orig_init = ml._initialize_adaptive_head

    def init_from_golden():
        orig_init()
        ml.adaptive_head.load_state_dict({v: torch.from_numpy(g["ml_before_" + v]) for v in NAMES.values()})
        ml.adaptive_head = ml.adaptive_head.to(ml.device)
    ml._initialize_adaptive_head = init_from_golden
    ml.add_examples(texts, labels)
    assert [ml.id_to_label[i] for i in range(3)] == g["ml_label_names"].tolist()
    tr = ml.last_training_trace
    assert tr["steps_per_epoch"] == g["ml_steps_per_epoch"].tolist()
    assert np.abs(np.array(tr["loss"]) - g["ml_loss"]).max() < 2e-3
    assert ml.label_thresholds == pytest.approx(json.loads(str(g["ml_thresholds"])))
    for t, ref in zip(g["ml_test_texts"].tolist(), g["ml_pred"].tolist()):
        ref = json.loads(ref)
        got = ml.predict_multilabel(t)
        assert [l for l, _ in got] == [l for l, _ in ref], (got, ref)
        assert np.allclose([s for _, s in got], [s for _, s in ref], atol=2e-3)
