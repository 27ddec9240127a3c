"""Textcat heads on the B200: the sm_100a textcat kernels against the fp32 ``TorchOps`` reference, and the
device-resident engine against the generic path for every textcat architecture."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _batch(lens, n_attr=4, vocab=40, seed=0):
    from spacy_ray_b200.nn.batch import make_token_batch

    rng = np.random.default_rng(seed)
    docs = [rng.integers(-vocab, vocab, size=(n, n_attr)).astype(np.int64) * 1000003 for n in lens]
    return make_token_batch(docs, device="cuda")


def _case(width, n_labels, lens, n_docs, *, seed=0, p_unknown=0.15):
    """bf16 tok2vec output (pad rows zero; docs 0 and 2 repeat one row: max-pooling ties), truths with
    unknown labels, bf16 weights as the flat buffer holds them."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    batch = _batch(lens, seed=seed)
    Tp = batch.n_rows
    X = torch.randn((Tp, width), generator=g, device="cuda")
    starts = batch.starts
    for d in (0, 2):
        if d < len(lens) and lens[d] > 1:
            X[starts[d]:starts[d] + lens[d]] = X[starts[d]]
    X = (X * batch.mask).to(torch.bfloat16)
    B = len(lens)
    truths = torch.rand((B, n_labels), generator=g, device="cuda").round()
    known = (torch.rand((B, n_labels), generator=g, device="cuda") >= p_unknown).float()
    truths[n_docs:] = 0
    known[n_docs:] = 0
    return batch, X, truths, known


def _weights(n_labels, P, bow_rows, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W = (torch.randn((n_labels, P), generator=g, device="cuda") * 0.2).to(torch.bfloat16) if P else None
    b = (torch.randn((n_labels,), generator=g, device="cuda") * 0.2).to(torch.bfloat16) if P else None
    Wb = (torch.randn((bow_rows, n_labels), generator=g, device="cuda") * 0.2).to(torch.bfloat16) if bow_rows else None
    bb = (torch.randn((n_labels,), generator=g, device="cuda") * 0.2).to(torch.bfloat16) if bow_rows else None
    return W, b, Wb, bb


def _check(width, n_labels, lens, n_docs, *, mean=True, mx=False, bow_rows=0, ngram=1, exclusive=True,
           no_output=False, neural=True, p_unknown=0.15):
    from spacy_ray_b200.ops.b200_ops import B200Ops
    from spacy_ray_b200.ops.torch_ops import TorchOps

    batch, X, truths, known = _case(width, n_labels, lens, n_docs, p_unknown=p_unknown)
    P = (int(mean) + int(mx)) * width if neural else 0
    W, b, Wb, bb = _weights(n_labels, P, bow_rows)
    if not neural:
        X = None
    kw = dict(use_mean=mean, use_max=mx, exclusive=exclusive, no_output_layer=no_output, ngram_size=ngram)
    ref = TorchOps(device="cuda", dtype=torch.float32)
    f32 = (lambda t: t.float() if t is not None else None)
    r_loss, r_scores, r_dX, r_g = ref.textcat_head(f32(X), batch, f32(W), f32(b), f32(Wb), f32(bb), truths, known,
                                                   n_docs=n_docs, **kw)
    ops = B200Ops("cuda:0")
    # gradients accumulate into what the buffers already hold
    pre = {k: torch.full_like(v, 0.5) for k, v in r_g.items()}
    go = {k: v.clone() for k, v in pre.items()}
    n_dev = torch.tensor([n_docs], dtype=torch.int32, device="cuda")
    loss, scores, dX, grads = ops.textcat_head(X, batch, W, b, Wb, bb, truths, known, n_docs=n_dev, grad_out=go,
                                               **kw)
    torch.cuda.synchronize()
    assert float(loss) == pytest.approx(float(r_loss), rel=2e-3, abs=1e-6)
    torch.testing.assert_close(scores, r_scores, rtol=2e-3, atol=2e-5)
    if neural:
        torch.testing.assert_close(dX.float(), r_dX.float(), rtol=2e-2, atol=1e-5)
        pad = batch.mask.reshape(-1) == 0
        assert torch.count_nonzero(dX[pad]) == 0, "pad rows of dX must stay exactly zero"
    for k, v in r_g.items():
        assert grads[k].data_ptr() == go[k].data_ptr()
        torch.testing.assert_close(grads[k] - pre[k], v, rtol=2e-3, atol=2e-5, msg=k)
    return batch, grads


@pytest.mark.parametrize("width", [32, 96, 256, 512])
@pytest.mark.parametrize("pool", ["mean", "max", "both"])
def test_textcat_kernels_match_the_reference(width, pool):
    lens = [5, 1, 7, 0, 300, 33, 2] + [11] * 40 + [0, 0, 0]       # partial batch: 47 real docs of 50 slots
    mean, mx = pool in ("mean", "both"), pool in ("max", "both")
    if (int(mean) + int(mx)) * width > 1024:
        pytest.skip("past the kernels' pooled-width limit (Trainer.unsupported_reason names it)")
    for n_labels in (1, 7, 128):
        _check(width, n_labels, lens, 47, mean=mean, mx=mx, exclusive=n_labels > 1)


@pytest.mark.parametrize("ngram", [1, 2, 3])
@pytest.mark.parametrize("variant", ["bow", "bow_no_output", "bow_logistic", "ensemble"])
def test_textcat_bow_kernels_match_the_reference(ngram, variant):
    lens = [4, 1, 0, 9, 200, 3, 3, 17] + [6] * 20 + [0, 0]
    neural = variant == "ensemble"
    for n_labels in (2, 33):
        _check(96, n_labels, lens, 28, mean=neural, bow_rows=262144, ngram=ngram, neural=neural,
               exclusive=variant != "bow_logistic", no_output=variant == "bow_no_output")


def test_bow_gradient_rows_are_the_hashed_ngrams():
    """The rows of the W_bow gradient that receive anything are exactly the feature indices
    ``models/textcat.py::_ngram_features`` names for the batch (an integer comparison)."""
    from spacy_ray_b200.models.textcat import _ngram_features

    lens = [4, 1, 9, 12, 3, 0, 8]
    batch, grads = _check(32, 3, lens, len(lens), mean=False, bow_rows=4096, ngram=3, neural=False,
                          p_unknown=0.0)
    batch.lengths = list(lens)
    batch.token_rows = None
    f, _d = _ngram_features(batch, 3, 4096)
    expected = torch.unique(f).cpu()
    got = torch.nonzero((grads["W_bow"] - 0.5).abs().sum(1) > 0).reshape(-1).cpu()
    assert torch.equal(got, expected)


def _worker(text):
    from spacy_ray_b200.config import Config
    from spacy_ray_b200.nn.layers import fix_random_seed
    from spacy_ray_b200.worker import Worker

    fix_random_seed(0)
    w = Worker(Config().from_str(text, interpolate=False), rank=0, num_workers=1, use_gpu=0, mode="sync",
               comm="auto")
    w.set_proxy(None)
    return w, list(w.train_corpus(w.nlp))


@pytest.mark.parametrize("arch,shared,multilabel", [
    ("cnn_mean", False, False), ("cnn_max", False, True), ("reduce_both", False, False), ("bow1", False, False),
    ("bow3", False, True), ("bow2_no_output", False, False), ("ensemble", False, False), ("ensemble", True, False),
    ("reduce_both", True, True)])
def test_engine_trains_textcat_like_the_generic_path(arch, shared, multilabel):
    """engine.Trainer (packed staging buffer -> CUDA-graph step) must give every head the losses of the
    generic nlp.update path on the same batches - textcat alone and next to NER on a shared tok2vec."""
    from test_textcat_engine import textcat_cfg

    from spacy_ray_b200.engine import Trainer

    text = textcat_cfg(arch, width=64, shared=shared, ner=shared, multilabel=multilabel, n_docs=300, max_len=16)
    bs, steps = 32, 12
    w_gen, exs = _worker(text)
    generic = []
    for step in range(steps):
        losses = {}
        w_gen.nlp.update(exs[step * 8: step * 8 + bs], drop=0.0, sgd=False, losses=losses)
        w_gen.proxy.step()
        generic.append({k: float(v) for k, v in losses.items()})
    w_fast, exs2 = _worker(text)
    trainer = Trainer(w_fast.nlp, w_fast.proxy, exs2, docs_per_batch=bs + 8, dropout=0.0, prefetch=False)
    fast = []
    for step in range(steps):
        trainer.prepare(np.arange(step * 8, step * 8 + bs))          # partial batches: 32 docs in 40 slots
        vec = trainer.step_async()
        fast.append({n: float(v) for n, v in trainer.losses_dict(vec).items()})
    assert len(trainer._graphs) >= 1
    trainer.close()
    heads = trainer.loss_names
    assert any(h.startswith("textcat") for h in heads) and (("ner" in heads) == shared)
    for g, f in zip(generic, fast):
        for head in heads:
            assert abs(g[head] - f[head]) <= 0.08 * abs(g[head]) + 0.02, (head, generic, fast)
    tc = [h for h in heads if h.startswith("textcat")][0]
    assert fast[-1][tc] < fast[0][tc]


def test_worker_trains_textcat_on_the_engine(tmp_path):
    from test_textcat_engine import textcat_cfg

    from spacy_ray_b200.config import Config
    from spacy_ray_b200.worker import Worker

    text = textcat_cfg("ensemble", width=64, shared=True, n_docs=1200, max_len=24)
    text = text.replace("max_steps = 10", "max_steps = 300").replace("eval_frequency = 5", "eval_frequency = 100")
    text += """
[training.batcher]
@batchers = "spacy.batch_by_sequence.v1"
size = 64
"""
    w = Worker(Config().from_str(text, interpolate=False), rank=0, num_workers=1, use_gpu=0, output_path=tmp_path)
    w.set_proxy(None)
    w.train(None, None)
    w.join(timeout=600)
    assert w.get_error() is None
    trainer = getattr(w.nlp, "_trainer", None)
    assert trainer is not None and trainer.steps >= 299, "the textcat pipeline did not run on the engine"
    scores = w.nlp.evaluate(list(w.dev_corpus(w.nlp)))
    assert scores["cats_score"] > 0.9, scores
