"""``spacy.TextCatCNN`` / ``spacy.TextCatReduce``: tok2vec -> pool over the tokens of each doc -> affine ->
softmax (exclusive classes) or logistic (multi-label).  The reference trains whatever spaCy pipeline the
config names (``/root/reference/spacy_ray/worker.py:88-96``); this is the document-level head of that zoo.

The pooled matrix is (n_docs, width) - tiny next to the token matrices - so it is built with plain
tensor ops from the padded-ragged layout (``nn/batch.py``); the affine layer is the shared ``Linear``.
``backprop`` takes the gradient w.r.t. the LOGITS (``probs - truth``, as ``Softmax`` does)."""
from __future__ import annotations

from typing import Optional

import torch

from ..nn.batch import TokenBatch
from ..nn.layers import Linear
from ..nn.model import Model


def _segments(batch: TokenBatch):
    lens = torch.as_tensor(batch.lengths, dtype=torch.int64, device=batch.device)
    seg = torch.repeat_interleave(torch.arange(len(batch.lengths), device=batch.device), lens)
    return lens, seg


def build_textcat_model(tok2vec: Model, exclusive_classes: bool = True, nO: Optional[int] = None,
                        use_reduce_mean: bool = True, use_reduce_max: bool = False, use_reduce_first: bool = False,
                        use_reduce_last: bool = False, ngram_size: Optional[int] = None,
                        no_output_layer: bool = False) -> Model:
    if use_reduce_first or use_reduce_last:
        raise ValueError("TextCat: only mean / max pooling are implemented (use_reduce_first / use_reduce_last are not)")
    if not (use_reduce_mean or use_reduce_max):
        raise ValueError("TextCat: enable use_reduce_mean and/or use_reduce_max")
    width = tok2vec.get_dim("nO")
    n_pool = int(use_reduce_mean) + int(use_reduce_max)
    output = Linear(nO, width * n_pool, init_zero=True, name="textcat_output")

    def init(model: Model, X=None, Y=None):
        tok2vec.initialize()
        if output.has_dim("nO") is None:
            if model.has_dim("nO") is None:
                raise ValueError("TextCat model: number of labels (nO) not set before initialize")
            output.set_dim("nO", model.get_dim("nO"))
        output.initialize()

    def forward(model: Model, batch: TokenBatch, is_train: bool):
        if not batch.lengths:
            raise ValueError("TextCat needs host-side doc lengths (generic path); it is not served by engine.Trainer")
        X, bp_t2v = tok2vec(batch, is_train)                       # (Tp, width), pad rows zero
        Xt = batch.unpad(X).float()                                # (T, width)
        lens, seg = _segments(batch)
        B = len(batch.lengths)
        inv = 1.0 / lens.clamp(min=1).to(torch.float32).unsqueeze(1)
        parts, ctx = [], {}
        if use_reduce_mean:
            sums = torch.zeros((B, width), dtype=torch.float32, device=X.device).index_add_(0, seg, Xt)
            parts.append(sums * inv)
        if use_reduce_max:
            mx = torch.full((B, width), float("-inf"), dtype=torch.float32, device=X.device)
            mx = mx.scatter_reduce(0, seg.unsqueeze(1).expand(-1, width), Xt, reduce="amax", include_self=True)
            mx = torch.where(torch.isinf(mx), torch.zeros_like(mx), mx)      # empty docs
            ctx["argmax"] = (Xt == mx[seg])
            parts.append(mx)
        pooled = torch.cat(parts, dim=1).to(X.dtype)
        logits, bp_out = output(pooled, is_train)
        logits = logits.float()
        scores = torch.softmax(logits, dim=1) if exclusive_classes else torch.sigmoid(logits)

        def backprop(d_logits: torch.Tensor):
            d_pooled = bp_out(d_logits.to(pooled.dtype)).float()
            dXt = torch.zeros_like(Xt)
            off = 0
            if use_reduce_mean:
                dXt += (d_pooled[:, off:off + width] * inv)[seg]
                off += width
            if use_reduce_max:
                hit = ctx["argmax"].float()
                hit = hit / hit.new_zeros((B, width)).index_add_(0, seg, hit).clamp(min=1.0)[seg]   # ties share
                dXt += d_pooled[:, off:off + width][seg] * hit
            bp_t2v(batch.pad(dXt.to(X.dtype)))
            return None

        return scores, backprop

    def update_with_cats(batch: TokenBatch, truths: torch.Tensor, known: torch.Tensor, n_docs):
        """Forward + loss + backward in one call (``ops.textcat_head``; works on device-resident batches
        without host lengths).  ``truths`` / ``known``: (B, nO) fp32; ``n_docs``: real doc count (int or
        a device int32 tensor).  Returns ``(loss, scores)``."""
        X, bp_t2v = tok2vec(batch, True)
        W, b = output.get_param("W"), output.get_param("b")
        go = {"W": output.grad_buffer("W"), "b": output.grad_buffer("b")} if getattr(model.ops, "fused", False) else None
        loss, scores, dX, grads = model.ops.textcat_head(
            X, batch, W, b, None, None, truths, known, n_docs=n_docs, use_mean=use_reduce_mean,
            use_max=use_reduce_max, exclusive=exclusive_classes, grad_out=go)
        output.inc_grad("W", grads["W"])
        output.inc_grad("b", grads["b"])
        bp_t2v(dX)
        return loss, scores

    model = Model("textcat", forward, init=init, dims={"nO": nO},
                  layers=[tok2vec, output], refs={"tok2vec": tok2vec, "output": output})
    model.attrs["exclusive_classes"] = bool(exclusive_classes)
    model.attrs["update_with_cats"] = update_with_cats
    return model


# ----------------------------------------------------------------------------------------------
# spacy.TextCatBOW / spacy.TextCatEnsemble: the architectures `spacy init config` writes for textcat
# ----------------------------------------------------------------------------------------------
def _ngram_features(batch: TokenBatch, ngram_size: int, length: int):
    """Hashed n-gram features (n = 1..ngram_size) of the NORM ids of every doc: ``(feature index, doc index)``
    pairs.  An n-gram never crosses a doc boundary."""
    ids = batch.unpad(batch.attrs[:, 0])                           # (T,) int64 hashed NORM ids
    _lens, seg = _segments(batch)
    feats, docs = [], []
    key = ids
    feats.append(key)
    docs.append(seg)
    for n in range(2, max(1, int(ngram_size)) + 1):
        if ids.numel() < n:
            break
        key = key[:-1] * 1000003 + ids[n - 1:]                     # int64 wrap-around is fine: it is a hash
        same = seg[: key.numel()] == seg[n - 1:]
        feats.append(key[same])
        docs.append(seg[: key.numel()][same])
    f = torch.cat(feats)
    f = (f ^ (f >> 31)).remainder(length)
    return f, torch.cat(docs)


def build_textcat_bow(exclusive_classes: bool = True, ngram_size: int = 1, no_output_layer: bool = False,
                      nO: Optional[int] = None, length: int = 262144) -> Model:
    """Sparse linear bag of n-grams (thinc ``SparseLinear``): ``scores[d] = sum_f W[f] + b`` over the hashed
    n-gram features ``f`` of doc ``d``, then softmax / logistic unless ``no_output_layer``."""

    def init(model: Model, X=None, Y=None):
        if model.has_param("W") is not True:
            n = model.get_dim("nO")
            model.set_param("W", model.ops.alloc((int(length), n), dtype=torch.float32))
            model.set_param("b", model.ops.alloc((n,), dtype=torch.float32))

    def forward(model: Model, batch: TokenBatch, is_train: bool):
        if not batch.lengths:
            raise ValueError("TextCatBOW needs host-side doc lengths (generic path)")
        W, b = model.get_param("W"), model.get_param("b")
        f, d = _ngram_features(batch, ngram_size, int(W.shape[0]))
        B = len(batch.lengths)
        logits = torch.zeros((B, W.shape[1]), dtype=torch.float32, device=W.device).index_add_(0, d, W.float()[f])
        logits = logits + b.float()
        if no_output_layer:
            scores = logits
        else:
            scores = torch.softmax(logits, dim=1) if exclusive_classes else torch.sigmoid(logits)

        def backprop(d_logits: torch.Tensor):
            d_logits = d_logits.float()
            dW = torch.zeros(W.shape, dtype=torch.float32, device=W.device).index_add_(0, f, d_logits[d])
            model.inc_grad("W", dW.to(W.dtype))
            model.inc_grad("b", d_logits.sum(0).to(b.dtype))
            return None

        return scores, backprop

    def update_with_cats(batch: TokenBatch, truths: torch.Tensor, known: torch.Tensor, n_docs):
        """Forward + loss + backward in one call (``ops.textcat_head``); see ``build_textcat_model``."""
        W, b = model.get_param("W"), model.get_param("b")
        go = {"W_bow": model.grad_buffer("W"), "b_bow": model.grad_buffer("b")} if getattr(model.ops, "fused", False) else None
        loss, scores, _dX, grads = model.ops.textcat_head(
            None, batch, None, None, W, b, truths, known, n_docs=n_docs, use_mean=False, use_max=False,
            exclusive=exclusive_classes, no_output_layer=no_output_layer, ngram_size=ngram_size, grad_out=go)
        model.inc_grad("W", grads["W_bow"])
        model.inc_grad("b", grads["b_bow"])
        return loss, scores

    model = Model("textcat_bow", forward, init=init, dims={"nO": nO}, params={"W": None, "b": None})
    model.attrs["exclusive_classes"] = bool(exclusive_classes)
    model.attrs["no_output_layer"] = bool(no_output_layer)
    model.attrs["ngram_size"] = int(ngram_size)
    model.attrs["update_with_cats"] = update_with_cats
    return model


def build_textcat_ensemble(tok2vec: Model, linear_model: Model, nO: Optional[int] = None) -> Model:
    """``spacy.TextCatEnsemble.v2``: a neural branch (tok2vec -> mean pool -> affine) and the sparse bag-of-words
    branch; here their LOGITS are added before the softmax / logistic (upstream concatenates the two score
    vectors and learns one more affine layer on top - same inputs, one layer less)."""
    exclusive = bool(linear_model.attrs.get("exclusive_classes", True))
    neural = build_textcat_model(tok2vec, exclusive_classes=exclusive, nO=nO)
    neural_out = neural.get_ref("output")
    t2v = neural.get_ref("tok2vec")

    def init(model: Model, X=None, Y=None):
        n = model.get_dim("nO")
        for m in (neural, linear_model):
            if m.has_dim("nO") is None:
                m.set_dim("nO", n)
        neural.initialize()
        linear_model.initialize()

    def forward(model: Model, batch: TokenBatch, is_train: bool):
        W, b = linear_model.get_param("W"), linear_model.get_param("b")
        f, d = _ngram_features(batch, int(linear_model.attrs.get("ngram_size", 1)), int(W.shape[0]))
        B = len(batch.lengths)
        bow = torch.zeros((B, W.shape[1]), dtype=torch.float32, device=W.device).index_add_(0, d, W.float()[f]) + b.float()
        X, bp_t2v = t2v(batch, is_train)
        Xt = batch.unpad(X).float()
        lens, seg = _segments(batch)
        inv = 1.0 / lens.clamp(min=1).to(torch.float32).unsqueeze(1)
        pooled = (torch.zeros((B, Xt.shape[1]), dtype=torch.float32, device=X.device).index_add_(0, seg, Xt) * inv).to(X.dtype)
        cnn, bp_out = neural_out(pooled, is_train)
        logits = cnn.float() + bow
        scores = torch.softmax(logits, dim=1) if exclusive else torch.sigmoid(logits)

        def backprop(d_logits: torch.Tensor):
            d_logits = d_logits.float()
            dW = torch.zeros(W.shape, dtype=torch.float32, device=W.device).index_add_(0, f, d_logits[d])
            linear_model.inc_grad("W", dW.to(W.dtype))
            linear_model.inc_grad("b", d_logits.sum(0).to(b.dtype))
            d_pooled = bp_out(d_logits.to(pooled.dtype)).float()
            bp_t2v(batch.pad(((d_pooled * inv)[seg]).to(X.dtype)))
            return None

        return scores, backprop

    def update_with_cats(batch: TokenBatch, truths: torch.Tensor, known: torch.Tensor, n_docs):
        """Forward + loss + backward in one call (``ops.textcat_head``); see ``build_textcat_model``.
        Gradients are handed over in the order the generic backward completes them: the bag of words,
        the output layer, then the tok2vec."""
        X, bp_t2v = t2v(batch, True)
        W, b = neural_out.get_param("W"), neural_out.get_param("b")
        Wb, bb = linear_model.get_param("W"), linear_model.get_param("b")
        go = None
        if getattr(model.ops, "fused", False):
            go = {"W": neural_out.grad_buffer("W"), "b": neural_out.grad_buffer("b"),
                  "W_bow": linear_model.grad_buffer("W"), "b_bow": linear_model.grad_buffer("b")}
        loss, scores, dX, grads = model.ops.textcat_head(
            X, batch, W, b, Wb, bb, truths, known, n_docs=n_docs, use_mean=True, use_max=False, exclusive=exclusive,
            ngram_size=int(linear_model.attrs.get("ngram_size", 1)), grad_out=go)
        linear_model.inc_grad("W", grads["W_bow"])
        linear_model.inc_grad("b", grads["b_bow"])
        neural_out.inc_grad("W", grads["W"])
        neural_out.inc_grad("b", grads["b"])
        bp_t2v(dX)
        return loss, scores

    model = Model("textcat_ensemble", forward, init=init, dims={"nO": nO},
                  layers=[neural, linear_model], refs={"tok2vec": t2v, "output": neural_out, "linear_model": linear_model})
    model.attrs["exclusive_classes"] = exclusive
    model.attrs["update_with_cats"] = update_with_cats
    return model
