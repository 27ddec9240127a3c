"""Textcat heads in the device-resident engine, host side: the packed staging buffer's per-document truths,
which configurations ``Trainer.unsupported_reason`` serves, ``TorchOps.textcat_head`` against the generic
forward / backward of every textcat architecture, and the synthetic corpus' textcat tasks."""
import numpy as np
import pytest
import torch

from spacy_ray_b200.config import Config
from spacy_ray_b200.pipeline.doc import Doc, Example

T2V_OWN = """
[components.{name}.model.tok2vec]
@architectures = "spacy.HashEmbedCNN.v2"
width = {width}
depth = 1
embed_size = 300
window_size = 1
maxout_pieces = 3
subword_features = true
pretrained_vectors = null
"""

T2V_LISTENER = """
[components.{name}.model.tok2vec]
@architectures = "spacy.Tok2VecListener.v1"
width = {width}
upstream = "*"
"""

SHARED_T2V = """
[components.tok2vec]
factory = "tok2vec"

[components.tok2vec.model]
@architectures = "spacy.HashEmbedCNN.v2"
width = {width}
depth = 1
embed_size = 300
window_size = 1
maxout_pieces = 3
subword_features = true
pretrained_vectors = null
"""

NER = """
[components.ner]
factory = "ner"

[components.ner.model]
@architectures = "spacy.TransitionBasedParser.v2"
state_type = "ner"
extra_state_tokens = false
hidden_width = 64
maxout_pieces = 2
use_upper = true
"""

BOW = """
@architectures = "spacy.TextCatBOW.v2"
exclusive_classes = {exclusive}
ngram_size = {ngram}
no_output_layer = {no_output}
"""

ARCHS = ["cnn_mean", "cnn_max", "reduce_both", "bow1", "bow2", "bow3", "bow2_no_output", "ensemble"]


def textcat_cfg(arch, *, width=32, shared=False, ner=False, multilabel=False, n_docs=120, max_len=12, ngram=None):
    """A pipeline with one textcat head of architecture ``arch`` (own tok2vec, or listening to a shared
    ``tok2vec`` component), optionally next to an NER head, trained on the synthetic corpus."""
    name = "textcat_multilabel" if multilabel else "textcat"
    exclusive = "false" if multilabel else "true"
    t2v = (T2V_LISTENER if shared else T2V_OWN).format(name=name, width=width)
    comp = f"\n[components.{name}]\nfactory = \"{name}\"\nthreshold = 0.5\n\n[components.{name}.model]\n"
    if arch.startswith("bow"):
        n = ngram or int(arch[3])
        comp += BOW.format(exclusive=exclusive, ngram=n, no_output="true" if "no_output" in arch else "false")
    elif arch == "ensemble":
        comp += "@architectures = \"spacy.TextCatEnsemble.v2\"\n" + t2v
        comp += f"\n[components.{name}.model.linear_model]\n" + BOW.format(exclusive=exclusive, ngram=ngram or 2,
                                                                           no_output="false")
    else:
        mean = "false" if arch == "cnn_max" else "true"
        mx = "true" if arch in ("cnn_max", "reduce_both") else "false"
        comp += (f"@architectures = \"spacy.TextCatReduce.v1\"\nexclusive_classes = {exclusive}\n"
                 f"use_reduce_mean = {mean}\nuse_reduce_max = {mx}\nuse_reduce_first = false\n"
                 f"use_reduce_last = false\n") + t2v
    pipeline = (["tok2vec"] if shared else []) + (["ner"] if ner else []) + [name]
    parts = [SHARED_T2V.format(width=width)] if shared else []
    if ner:
        parts.append(NER + (T2V_LISTENER if shared else T2V_OWN).format(name="ner", width=width))
    parts.append(comp)
    tasks = (["ner"] if ner else []) + [name]
    corpus = "".join(f"""
[corpora.{split}]
@readers = "spacy_ray_b200.SyntheticCorpus.v1"
n_docs = {n}
seed = {seed}
min_len = 2
max_len = {max_len}
vocab_size = 60
tasks = {tasks!r}
""" for split, n, seed in (("train", n_docs, 1), ("dev", 60, 2)))
    return (f"[nlp]\nlang = \"en\"\npipeline = {pipeline!r}\n\n[components]\n" + "".join(parts) + "\n[corpora]\n"
            + corpus + "\n[training]\nmax_steps = 10\neval_frequency = 5\ndropout = 0.0\n").replace("'", '"')


def _nlp(text):
    from spacy_ray_b200.nn.layers import fix_random_seed
    from spacy_ray_b200.pipeline.language import Language
    from spacy_ray_b200.training.corpus import create_synthetic_corpus

    fix_random_seed(0)
    cfg = Config().from_str(text, interpolate=False)
    nlp = Language.from_config(cfg)
    tr = {k: v for k, v in cfg["corpora"]["train"].items() if not k.startswith("@")}
    examples = list(create_synthetic_corpus(**tr)())
    nlp.initialize(lambda: examples)
    return nlp, examples


def _head(nlp):
    return [(n, c) for n, c in nlp.pipeline if n.startswith("textcat")][0]


def _grads(model):
    out = {}
    for i, node in enumerate(model.walk()):
        for p in node.param_names:
            if node.has_grad(p):
                out[(i, node.name, p)] = node.get_grad(p).clone().float()
    return out


def _clear(model):
    for node in model.walk():
        node._params.clear_grads()


def _randomise(model):
    """Non-zero output layers (they are zero-initialised) so every gradient path carries signal."""
    g = torch.Generator().manual_seed(7)
    for node in model.walk():
        if node.name in ("textcat_output", "textcat_bow"):
            for p in node.param_names:
                if node.has_param(p):
                    v = node.get_param(p)
                    v.copy_(torch.randn(v.shape, generator=g) * 0.5)


def _special_docs():
    """Max-pooling ties (a repeated word: identical window features in the middle), a length-0 doc, a
    length-1 doc, and a doc with a label missing from its cats."""
    return [Doc(["aa", "aa", "aa", "aa", "aa"], cats={"MARKED": 1.0, "PLAIN": 0.0}),
            Doc([], cats={"MARKED": 0.0, "PLAIN": 1.0}),
            Doc(["zz"], cats={"MARKED": 1.0, "PLAIN": 0.0}),
            Doc(["x", "y", "x", "y"], cats={"PLAIN": 1.0})]


@pytest.mark.parametrize("arch", ARCHS)
def test_torch_textcat_head_matches_the_generic_model(arch):
    """``update_with_cats`` (TorchOps.textcat_head, device-side doc lengths) must give the generic forward /
    backward's loss, scores and every parameter gradient - the tok2vec's included, so dX too."""
    nlp, examples = _nlp(textcat_cfg(arch))
    name, comp = _head(nlp)
    _randomise(comp.model)
    egs = examples[:9] + [Example.from_doc(d) for d in _special_docs()]
    batch = nlp.make_batch([eg.predicted for eg in egs])
    _clear(comp.model)
    losses = {}
    scores_g = comp.model.predict(batch)
    comp.update(egs, batch=batch, drop=0.0, sgd=False, losses=losses)
    g_generic = _grads(comp.model)
    _clear(comp.model)
    truths, known = comp._truths(egs, "cpu")
    loss, scores = comp.model.attrs["update_with_cats"](batch, truths, known, len(egs))
    g_fast = _grads(comp.model)
    assert float(loss) == pytest.approx(float(losses[name]), rel=1e-5, abs=1e-7)
    torch.testing.assert_close(scores.float(), scores_g.float(), rtol=1e-5, atol=1e-6)
    assert g_fast.keys() == g_generic.keys() and g_fast
    for key in g_generic:
        torch.testing.assert_close(g_fast[key], g_generic[key], rtol=1e-4, atol=1e-6, msg=str(key))


def test_torch_textcat_head_ignores_doc_slots_past_the_batch():
    """A partial batch (doc slots past ``n_docs``, as the engine's fixed-capacity buffer has them) computes
    exactly what the batch of the real docs alone computes."""
    from spacy_ray_b200.ops import get_current_ops

    nlp, examples = _nlp(textcat_cfg("reduce_both"))
    _name, comp = _head(nlp)
    _randomise(comp.model)
    ops = get_current_ops()
    out = comp.model.get_ref("output")
    W, b = out.get_param("W"), out.get_param("b")
    egs = examples[:6]
    truths, known = comp._truths(egs, "cpu")
    full = nlp.make_batch([eg.predicted for eg in egs])
    X = torch.randn((full.n_rows, 32), generator=torch.Generator().manual_seed(3)) * full.mask
    ref = ops.textcat_head(X, full, W, b, None, None, truths, known, use_mean=True, use_max=True)
    padded = nlp.make_batch([eg.predicted for eg in egs] + [eg.predicted for eg in examples[6:9]])
    Xp = torch.zeros((padded.n_rows, 32))
    Xp[: full.n_rows] = X
    tp = torch.cat([truths, torch.zeros((3, truths.shape[1]))])
    kp = torch.cat([known, torch.zeros((3, truths.shape[1]))])
    got = ops.textcat_head(Xp, padded, W, b, None, None, tp, kp, n_docs=torch.tensor([6], dtype=torch.int32),
                           use_mean=True, use_max=True)
    assert float(got[0]) == pytest.approx(float(ref[0]))
    torch.testing.assert_close(got[1][:6], ref[1])
    assert torch.count_nonzero(got[1][6:]) == 0
    torch.testing.assert_close(got[2][: full.n_rows], ref[2])
    assert torch.count_nonzero(got[2][full.n_rows:]) == 0
    for k in ref[3]:
        torch.testing.assert_close(got[3][k], ref[3][k])


def test_torch_ngram_features_equal_the_generic_hash():
    from spacy_ray_b200.models.textcat import _ngram_features
    from spacy_ray_b200.ops.torch_ops import TorchOps

    nlp, examples = _nlp(textcat_cfg("bow3"))
    batch = nlp.make_batch([eg.predicted for eg in examples[:20]] + [Doc([]), Doc(["q"])])
    batch.attrs[:, 0] = batch.attrs[:, 0] * 7919 - (1 << 62)           # ids across the whole int64 range
    for n in (1, 2, 3):
        f, d = _ngram_features(batch, n, 262144)
        lens = batch.doc_lens.long()
        seg = torch.repeat_interleave(torch.arange(lens.numel()), lens)
        f2, d2 = TorchOps._ngram_features(batch.unpad(batch.attrs[:, 0]), seg, n, 262144)
        assert torch.equal(f, f2) and torch.equal(d, d2)


def test_staging_buffer_carries_the_cats_of_full_and_partial_batches():
    from spacy_ray_b200.engine.trainer import ExampleStore, _kind, _Layout, fill_stage, make_stage

    nlp, examples = _nlp(textcat_cfg("cnn_mean", ner=True))
    # labels missing from some docs stay "unknown"
    for eg in examples[::3]:
        eg.reference.cats = {"PLAIN": eg.reference.cats["PLAIN"]}
    name, comp = _head(nlp)
    heads = [(n, c, _kind(c)) for n, c in nlp.pipeline if getattr(c, "is_trainable", False)]
    assert [k for _n, _c, k in heads] == ["ner", "textcat"]
    store = ExampleStore(examples, heads)
    B = 16
    lay = _Layout(rows=512, docs=B, lmax=64, slots=tuple(store.slots), n_attr=int(store.attrs.shape[1]),
                  cats=tuple((k, int(t.shape[1])) for k, (t, _kn) in store.cats.items()))
    stage = make_stage(lay, store, pin=False)
    for ids in (np.arange(3, 3 + B), np.array([5, 0, 9, 2, 7])):
        fill_stage(store, lay, stage, ids)
        t, k = comp._truths([examples[i] for i in ids], "cpu")
        got_t, got_k = stage["np"]["cats"][name]
        n = len(ids)
        assert np.array_equal(got_t[:n], t.numpy()) and np.array_equal(got_k[:n], k.numpy())
        assert not got_t[n:].any() and not got_k[n:].any()
        assert int(stage["np"]["meta"][1]) == n
        assert (got_k[:n] == 0).any()


@pytest.mark.parametrize("arch,shared", [(a, False) for a in ARCHS] + [("cnn_mean", True), ("reduce_both", True),
                                                                         ("ensemble", True)])
def test_engine_serves_every_textcat_architecture(arch, shared):
    from spacy_ray_b200.engine.trainer import Trainer, _kind

    nlp, _ = _nlp(textcat_cfg(arch, shared=shared, ner=shared))
    _name, comp = _head(nlp)
    assert _kind(comp) == "textcat"
    assert Trainer.unsupported_reason(nlp) is None


def test_engine_serves_multilabel_textcat():
    from spacy_ray_b200.engine.trainer import Trainer, _kind

    nlp, _ = _nlp(textcat_cfg("reduce_both", multilabel=True))
    _name, comp = _head(nlp)
    assert _kind(comp) == "textcat" and Trainer.unsupported_reason(nlp) is None


@pytest.mark.parametrize("arch,kw,what", [("reduce_both", {"width": 768}, "pooled width"),
                                           ("bow1", {"ngram": 9}, "ngram_size")])
def test_engine_names_textcat_heads_past_the_kernel_limits(arch, kw, what):
    from spacy_ray_b200.engine.trainer import Trainer

    nlp, _ = _nlp(textcat_cfg(arch, **kw))
    why = Trainer.unsupported_reason(nlp)
    assert why is not None and why.startswith("textcat:") and what in why, why


def test_engine_names_textcat_heads_with_too_many_labels():
    from spacy_ray_b200.engine.trainer import Trainer

    nlp, examples = _nlp(textcat_cfg("bow1", multilabel=True))
    _name, comp = _head(nlp)
    for i in range(200):
        comp._labels.append(f"EXTRA{i}")
    why = Trainer.unsupported_reason(nlp)
    assert why is not None and "labels" in why, why


def test_synthetic_textcat_tasks_are_deterministic_and_leave_the_other_layers_alone():
    from spacy_ray_b200.training.corpus import SyntheticCorpus

    base = SyntheticCorpus(n_docs=80, seed=4, min_len=3, max_len=20, tasks=("tagger", "ner", "parser")).docs()
    for task in ("textcat", "textcat_multilabel"):
        a = SyntheticCorpus(n_docs=80, seed=4, min_len=3, max_len=20, tasks=("tagger", "ner", "parser", task)).docs()
        b = SyntheticCorpus(n_docs=80, seed=4, min_len=3, max_len=20, tasks=("tagger", "ner", "parser", task)).docs()
        for x, y, z in zip(a, b, base):
            assert x.words == z.words and x.tags == z.tags and x.ents == z.ents and x.heads == z.heads
            assert x.cats == y.cats and x.cats and not z.cats
        values = np.array([list(d.cats.values()) for d in a])
        assert 0.2 < values[:, 0].mean() < 0.8                           # both outcomes occur
        if task == "textcat":
            assert np.all(values.sum(axis=1) == 1.0)
    with pytest.raises(ValueError):
        SyntheticCorpus(tasks=("textcat", "textcat_multilabel"))
