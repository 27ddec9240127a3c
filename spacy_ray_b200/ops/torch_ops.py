"""Reference backend: every op as plain PyTorch.

Each method documents the exact math; the sm_100a kernels in ``ops/csrc`` are
tested against these (fp32).  The op set is the transitive hot path of the
reference - what thinc's ``CupyOps`` runs when spacy-ray trains (SURVEY.md
section 2.7, K1-K9): hashing + HashEmbed gather, Maxout, LayerNorm,
expand_window (seq2col), residual/dropout, softmax cross-entropy, Adam.

Batch layout ("padded ragged"): all docs of a batch are flattened into one
``(Tp, width)`` array with **one all-zero row before the first doc, between
consecutive docs and after the last doc**.  ``mask`` is ``(Tp, 1)``, 1.0 on
real tokens.  Because pad rows are kept at exactly zero by every layer,
``expand_window`` needs no per-doc logic: neighbours at a doc edge read the
zero row.  (On the GPU the same trick lets a TMA load at row offset -1/0/+1
feed the window GEMM without materialising the ``(T, 3*width)`` array.)
"""
from __future__ import annotations

import math
from typing import Any, Dict, List, Optional, Sequence, Tuple

import torch

_M64 = (1 << 64) - 1


def _s64(x: int) -> int:
    """Python int -> the signed 64-bit value with the same bit pattern."""
    x &= _M64
    return x - (1 << 64) if x >= (1 << 63) else x


_GOLDEN = 0x9E3779B97F4A7C15
_FMIX1 = 0xFF51AFD7ED558CCD
_FMIX2 = 0xC4CEB9FE1A85EC53


def fmix64_int(h: int) -> int:
    """MurmurHash3 64-bit finaliser on Python ints (ground truth for tests)."""
    h &= _M64
    h ^= h >> 33
    h = (h * _FMIX1) & _M64
    h ^= h >> 33
    h = (h * _FMIX2) & _M64
    h ^= h >> 33
    return h


def hash_rows_int(attr_id: int, seed: int, n_rows: int) -> Tuple[int, int, int, int]:
    """The four table rows a 64-bit attribute id maps to (pure Python)."""
    h1 = fmix64_int((attr_id & _M64) ^ ((seed * _GOLDEN) & _M64))
    h2 = fmix64_int((h1 + _GOLDEN) & _M64)
    return (
        (h1 & 0xFFFFFFFF) % n_rows,
        (h1 >> 32) % n_rows,
        (h2 & 0xFFFFFFFF) % n_rows,
        (h2 >> 32) % n_rows,
    )


def _lsr(x: torch.Tensor, s: int) -> torch.Tensor:
    """Logical shift right on int64 tensors (torch's ``>>`` is arithmetic)."""
    return (x >> s) & ((1 << (64 - s)) - 1)


def _fmix64(h: torch.Tensor) -> torch.Tensor:
    h = h ^ _lsr(h, 33)
    h = h * _s64(_FMIX1)
    h = h ^ _lsr(h, 33)
    h = h * _s64(_FMIX2)
    h = h ^ _lsr(h, 33)
    return h


class TorchOps:
    name = "torch"
    fused = False

    def __init__(self, device: str = "cpu", dtype: torch.dtype = torch.float32):
        self.device = torch.device(device)
        self.dtype = dtype          # parameter / activation dtype
        self.device_type = self.device.type

    # ------------------------------------------------------------------ alloc
    def alloc(self, shape, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
        return torch.zeros(shape, dtype=dtype or self.dtype, device=self.device)

    def asarray(self, data, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
        t = torch.as_tensor(data)
        if dtype is None and t.is_floating_point():
            dtype = self.dtype
        return t.to(device=self.device, dtype=dtype) if dtype is not None else t.to(self.device)

    def to_host(self, t: torch.Tensor) -> torch.Tensor:
        return t.detach().to("cpu")

    # ------------------------------------------------------------------ init
    def glorot_uniform(self, shape: Sequence[int], fan_in: int, fan_out: int, gen: torch.Generator) -> torch.Tensor:
        scale = math.sqrt(6.0 / float(fan_in + fan_out))
        w = (torch.rand(tuple(shape), generator=gen, dtype=torch.float32) * 2 - 1) * scale
        return w.to(device=self.device, dtype=self.dtype)

    def uniform(self, shape: Sequence[int], lo: float, hi: float, gen: torch.Generator) -> torch.Tensor:
        w = torch.rand(tuple(shape), generator=gen, dtype=torch.float32) * (hi - lo) + lo
        return w.to(device=self.device, dtype=self.dtype)

    # ------------------------------------------------------------------ K1 hashing / HashEmbed
    def hash_rows(self, ids: torch.Tensor, seed: int, n_rows: int) -> torch.Tensor:
        """``ids`` ``(N,)`` int64 (bit pattern of a uint64 attribute id) ->
        ``(N, 4)`` int64 row indices in ``[0, n_rows)``.

        h1 = fmix64(id ^ seed*GOLDEN); h2 = fmix64(h1 + GOLDEN);
        rows = [lo32(h1), hi32(h1), lo32(h2), hi32(h2)] % n_rows."""
        ids = ids.to(torch.int64)
        h1 = _fmix64(ids ^ _s64(seed * _GOLDEN))
        h2 = _fmix64(h1 + _s64(_GOLDEN))
        parts = [h1 & 0xFFFFFFFF, _lsr(h1, 32), h2 & 0xFFFFFFFF, _lsr(h2, 32)]
        return torch.stack(parts, dim=1) % n_rows

    def multi_hash_embed(
        self,
        attrs: torch.Tensor,
        mask: torch.Tensor,
        tables: Sequence[torch.Tensor],
        seeds: Sequence[int],
        columns: Sequence[int],
    ) -> torch.Tensor:
        """For each table a: ``Y[:, a*nO:(a+1)*nO] = mask * sum_k E_a[rows_a[:, k]]``
        - the concatenated output of the four HashEmbed layers."""
        outs = []
        for E, seed, col in zip(tables, seeds, columns):
            rows = self.hash_rows(attrs[:, col], seed, E.shape[0])
            outs.append(E[rows].to(torch.float32).sum(dim=1))
        Y = torch.cat(outs, dim=1) * mask.to(torch.float32)
        return Y.to(self.dtype)

    def multi_hash_embed_backward(
        self,
        dY: torch.Tensor,
        attrs: torch.Tensor,
        mask: torch.Tensor,
        n_rows: Sequence[int],
        seeds: Sequence[int],
        columns: Sequence[int],
        out: Optional[Sequence[torch.Tensor]] = None,
        perm: Optional[torch.Tensor] = None,     # rows pre-grouped by id (used by the CUDA backend)
    ) -> List[torch.Tensor]:
        """``dE_a[rows_a[t, k]] += mask[t] * dY[t, a-block]`` for k in 0..3 (fp32)."""
        dY = dY.to(torch.float32) * mask.to(torch.float32)
        nO = dY.shape[1] // len(n_rows)
        grads = []
        for a, (nV, seed, col) in enumerate(zip(n_rows, seeds, columns)):
            rows = self.hash_rows(attrs[:, col], seed, nV)
            dE = out[a] if out is not None else torch.zeros((nV, nO), dtype=torch.float32, device=dY.device)
            block = dY[:, a * nO:(a + 1) * nO]
            for k in range(4):
                dE.index_add_(0, rows[:, k], block)
            grads.append(dE)
        return grads

    # ------------------------------------------------------------------ K4 expand_window in padded layout
    def seq2col(self, X: torch.Tensor, window: int) -> torch.Tensor:
        """``(Tp, nI) -> (Tp, (2*window+1)*nI)``: [X[t-w] ... X[t] ... X[t+w]], rows
        outside the array read as zero.  Doc boundaries are handled by the zero
        pad rows of the batch layout."""
        if window == 0:
            return X
        cols = []
        Tp = X.shape[0]
        for off in range(-window, window + 1):
            if off == 0:
                cols.append(X)
                continue
            shifted = torch.zeros_like(X)
            if off < 0:
                shifted[-off:] = X[: Tp + off]
            else:
                shifted[: Tp - off] = X[off:]
            cols.append(shifted)
        return torch.cat(cols, dim=1)

    def backprop_seq2col(self, dXw: torch.Tensor, window: int) -> torch.Tensor:
        if window == 0:
            return dXw
        n = 2 * window + 1
        nI = dXw.shape[1] // n
        Tp = dXw.shape[0]
        dX = torch.zeros((Tp, nI), dtype=dXw.dtype, device=dXw.device)
        for j, off in enumerate(range(-window, window + 1)):
            block = dXw[:, j * nI:(j + 1) * nI]
            if off == 0:
                dX += block
            elif off < 0:
                dX[: Tp + off] += block[-off:]
            else:
                dX[off:] += block[: Tp - off]
        return dX

    # ------------------------------------------------------------------ dropout
    def dropout_mask(self, seed: int, n_rows: int, n_cols: int, p: float) -> torch.Tensor:
        """Counter-based Bernoulli mask, scaled by 1/(1-p).  Elements are hashed in groups of
        four: ``h = fmix64(seed*GOLDEN + (idx >> 2))`` with ``idx = r*n_cols + c``; element ``idx``
        takes bits ``16*(idx & 3) .. +16`` of ``h`` and is kept iff that value ``>= floor(p * 2^16)``
        (float32 product, as the kernels compute it).  Stateless, so a CUDA kernel regenerates
        the same mask in backward."""
        import numpy as np

        idx = torch.arange(n_rows * n_cols, dtype=torch.int64, device=self.device)
        h = _fmix64((idx >> 2) + _s64(seed * _GOLDEN))
        u = (h >> (16 * (idx & 3))) & 0xFFFF      # sign extension only touches the masked-off bits
        thr = int(np.float32(p) * np.float32(65536.0))
        keep = (u >= thr).to(torch.float32) * (1.0 / (1.0 - p))
        return keep.view(n_rows, n_cols)

    # ------------------------------------------------------------------ K2+K3+K4+K5 fused block
    def maxout_block(
        self,
        X: torch.Tensor,
        W: torch.Tensor,
        b: torch.Tensor,
        G: Optional[torch.Tensor],
        beta: Optional[torch.Tensor],
        mask: torch.Tensor,
        *,
        window: int = 0,
        residual: bool = False,
        dropout: float = 0.0,
        is_train: bool = False,
        seed: int = 0,
    ) -> Tuple[torch.Tensor, Dict[str, Any]]:
        """One tok2vec block.

        Xw = seq2col(X, window); Z = Xw @ W.view(nO*nP, nI)^T + b;
        H = max_p Z[:, o, p], which = argmax_p;
        N = (H - mean) / sqrt(var + 1e-8) * G + beta      (if G is given)
        D = N * dropout_mask                               (training only)
        Y = mask * (X + D  if residual else  D)
        """
        nO, nP, nI = W.shape
        Xf = X.to(torch.float32)
        Xw = self.seq2col(Xf, window)
        Z = Xw @ W.to(torch.float32).reshape(nO * nP, nI).t() + b.to(torch.float32).reshape(-1)
        H, which = Z.view(-1, nO, nP).max(dim=2)
        ctx: Dict[str, Any] = {
            "X": X, "W": W, "which": which.to(torch.uint8), "window": window, "residual": residual,
            "mask": mask, "nP": nP, "has_ln": G is not None,
        }
        if G is not None:
            mu = H.mean(dim=1, keepdim=True)
            var = H.var(dim=1, unbiased=False, keepdim=True) + 1e-8
            rstd = var.rsqrt()
            xhat = (H - mu) * rstd
            N = xhat * G.to(torch.float32) + beta.to(torch.float32)
            ctx.update({"xhat": xhat, "rstd": rstd, "G": G})
        else:
            N = H
        if is_train and dropout > 0.0:
            dm = self.dropout_mask(seed, N.shape[0], N.shape[1], dropout)
            N = N * dm
            ctx["dropmask"] = dm
        Y = (Xf + N) if residual else N
        Y = Y * mask.to(torch.float32)
        return Y.to(self.dtype), ctx

    def maxout_block_backward(self, dY: torch.Tensor, ctx: Dict[str, Any], grad_out=None):
        """Returns ``(dX, dW, db, dG, dbeta)`` (fp32; dG/dbeta None without LN)."""
        mask = ctx["mask"].to(torch.float32)
        dYm = dY.to(torch.float32) * mask
        dN = dYm
        if "dropmask" in ctx:
            dN = dN * ctx["dropmask"]
        if ctx["has_ln"]:
            xhat, rstd, G = ctx["xhat"], ctx["rstd"], ctx["G"].to(torch.float32)
            dG = (dN * xhat).sum(dim=0)
            dbeta = dN.sum(dim=0)
            dxh = dN * G
            dH = rstd * (dxh - dxh.mean(dim=1, keepdim=True) - xhat * (dxh * xhat).mean(dim=1, keepdim=True))
            # pad rows: dN is zero there so dH is zero too
        else:
            dG = dbeta = None
            dH = dN
        W = ctx["W"].to(torch.float32)
        nO, nP, nI = W.shape
        dZ = torch.zeros((dH.shape[0], nO, nP), dtype=torch.float32, device=dH.device)
        dZ.scatter_(2, ctx["which"].to(torch.int64).unsqueeze(2), dH.unsqueeze(2))
        dZ = dZ.view(-1, nO * nP)
        Xw = self.seq2col(ctx["X"].to(torch.float32), ctx["window"])
        dW = (dZ.t() @ Xw).view(nO, nP, nI)
        db = dZ.sum(dim=0).view(nO, nP)
        dXw = dZ @ W.reshape(nO * nP, nI)
        dX = self.backprop_seq2col(dXw, ctx["window"])
        if ctx["residual"]:
            dX = dX + dYm
        return dX, dW, db, dG, dbeta

    # ------------------------------------------------------------------ Linear
    def linear(self, X: torch.Tensor, W: torch.Tensor, b: Optional[torch.Tensor]) -> torch.Tensor:
        Y = X.to(torch.float32) @ W.to(torch.float32).t()
        if b is not None:
            Y = Y + b.to(torch.float32)
        return Y.to(self.dtype)

    def linear_backward(self, dY: torch.Tensor, X: torch.Tensor, W: torch.Tensor, need_dX: bool = True,
                        need_db: bool = True):
        dYf = dY.to(torch.float32)
        dW = dYf.t() @ X.to(torch.float32)
        db = dYf.sum(dim=0) if need_db else None
        dX = dYf @ W.to(torch.float32) if need_dX else None
        return dX, dW, db

    # ------------------------------------------------------------------ K6 softmax + cross-entropy
    def softmax(self, logits: torch.Tensor) -> torch.Tensor:
        return torch.softmax(logits.to(torch.float32), dim=-1)

    def softmax_xent(
        self,
        X: torch.Tensor,
        W: torch.Tensor,
        b: torch.Tensor,
        labels: torch.Tensor,
    ):
        """Tagger head.  ``logits = X @ W^T + b``; ``P = softmax(logits)``;
        for rows with ``labels >= 0``: ``d = P - onehot(label)`` else ``d = 0``;
        ``loss = sum(d**2)`` (the quantity spaCy's tagger reports).
        Returns ``(loss, d_logits, guesses, dX, dW, db)``."""
        Xf = X.to(torch.float32)
        logits = Xf @ W.to(torch.float32).t() + b.to(torch.float32)
        P = torch.softmax(logits, dim=-1)
        guesses = P.argmax(dim=-1)
        have = (labels >= 0)
        d = P.clone()
        idx = torch.nonzero(have, as_tuple=False).squeeze(1)
        d[idx, labels[idx]] -= 1.0
        d = d * have.unsqueeze(1).to(torch.float32)
        loss = (d * d).sum()
        dW = d.t() @ Xf
        db = d.sum(dim=0)
        dX = d @ W.to(torch.float32)
        return loss, d, guesses, dX, dW, db

    # ------------------------------------------------------------------ textcat head
    def textcat_head(self, X, batch, W, b, W_bow, b_bow, truths, known, *, n_docs=None, use_mean: bool = True,
                     use_max: bool = False, exclusive: bool = True, no_output_layer: bool = False,
                     ngram_size: int = 1, grad_out: Optional[Dict[str, torch.Tensor]] = None):
        """Forward + loss + backward of a textcat head over the docs of ``batch`` (device ``doc_starts`` /
        ``doc_lens``; slots ``>= n_docs`` are unused).  The math of ``models/textcat.py``:

        pooled = [mean | max over the doc's rows of X]; logits = pooled W^T + b (if ``W``)
                 + sum over the doc's hashed n-grams f of W_bow[f] + b_bow (if ``W_bow``);
        scores = softmax (exclusive) | logistic | identity (``no_output_layer``);
        diff = (scores - truths) * known; loss = mean(diff^2) over (n_docs, n_labels);
        d_logits = diff / n_docs; dX: mean -> d / len, max -> d * [x == max] / n_ties.

        ``n_docs``: int or a 1-element int tensor (None: every slot is a doc).  Gradients are accumulated
        into ``grad_out[name]`` when given (names ``W``, ``b``, ``W_bow``, ``b_bow``), else fresh tensors.
        Returns ``(loss, scores, dX, grads)``; ``dX`` is None without ``X``."""
        dev = truths.device
        lens = batch.doc_lens.to(device=dev, dtype=torch.int64)
        starts = batch.doc_starts.to(device=dev, dtype=torch.int64)
        B = int(lens.numel())
        n = B if n_docs is None else int(torch.as_tensor(n_docs).reshape(-1)[0])
        valid = (torch.arange(B, device=dev) < n)
        lens = torch.where(valid, lens, torch.zeros_like(lens))
        seg = torch.repeat_interleave(torch.arange(B, device=dev), lens)
        rows = starts[seg] + (torch.arange(int(lens.sum()), device=dev) - (torch.cumsum(lens, 0) - lens)[seg])
        nL = int(truths.shape[1])
        logits = torch.zeros((B, nL), dtype=torch.float32, device=dev)
        ctx = {}
        if X is not None:
            width = X.shape[1]
            Xt = X.index_select(0, rows).to(torch.float32)
            inv = 1.0 / lens.clamp(min=1).to(torch.float32).unsqueeze(1)
            parts = []
            if use_mean:
                parts.append(torch.zeros((B, width), dtype=torch.float32, device=dev).index_add_(0, seg, Xt) * inv)
            if use_max:
                mx = torch.full((B, width), float("-inf"), dtype=torch.float32, device=dev)
                mx = mx.scatter_reduce(0, seg.unsqueeze(1).expand(-1, width), Xt, reduce="amax", include_self=True)
                mx = torch.where(torch.isinf(mx), torch.zeros_like(mx), mx)
                ctx["argmax"] = (Xt == mx[seg])
                parts.append(mx)
            pooled = torch.cat(parts, dim=1)
            logits = logits + pooled @ W.to(torch.float32).t() + b.to(torch.float32)
        f = d = None
        if W_bow is not None:
            f, d = self._ngram_features(batch.attrs[:, 0].to(dev).index_select(0, rows), seg, ngram_size,
                                        int(W_bow.shape[0]))
            logits = logits.index_add(0, d, W_bow.to(torch.float32)[f]) + b_bow.to(torch.float32)
        if no_output_layer:
            scores = logits
        else:
            scores = torch.softmax(logits, dim=1) if exclusive else torch.sigmoid(logits)
        scores = scores * valid.unsqueeze(1)
        diff = (scores - truths.to(torch.float32)) * known.to(torch.float32) * valid.unsqueeze(1)
        loss = (diff * diff).sum() / (max(n, 1) * nL)
        d_logits = diff / max(n, 1)
        go = grad_out or {}

        def acc(name, value):
            buf = go.get(name)
            if buf is None:
                return value
            buf.view(value.shape).add_(value.to(buf.dtype))
            return buf

        grads: Dict[str, torch.Tensor] = {}
        dX = None
        if W_bow is not None:
            grads["W_bow"] = acc("W_bow", torch.zeros((W_bow.shape[0], nL), dtype=torch.float32, device=dev)
                                 .index_add_(0, f, d_logits[d]))
            grads["b_bow"] = acc("b_bow", d_logits.sum(0))
        if X is not None:
            grads["W"] = acc("W", d_logits.t() @ pooled)
            grads["b"] = acc("b", d_logits.sum(0))
            d_pooled = d_logits @ W.to(torch.float32)
            dXt = torch.zeros_like(Xt)
            off = 0
            if use_mean:
                dXt += (d_pooled[:, off:off + width] * inv)[seg]
                off += width
            if use_max:
                hit = ctx["argmax"].to(torch.float32)
                hit = hit / hit.new_zeros((B, width)).index_add_(0, seg, hit).clamp(min=1.0)[seg]
                dXt += d_pooled[:, off:off + width][seg] * hit
            dX = torch.zeros(X.shape, dtype=torch.float32, device=dev)
            dX.index_copy_(0, rows, dXt)
            dX = dX.to(X.dtype)
        return loss, scores, dX, grads

    @staticmethod
    def _ngram_features(ids: torch.Tensor, seg: torch.Tensor, ngram_size: int, length: int):
        """``(feature index, doc index)`` of every n-gram (n = 1..ngram_size) of the token-order NORM ids
        ``ids`` (doc ``seg``): the hash of ``models/textcat.py::_ngram_features``."""
        feats, docs = [ids], [seg]
        key = ids
        for n in range(2, max(1, int(ngram_size)) + 1):
            if ids.numel() < n:
                break
            key = key[:-1] * 1000003 + ids[n - 1:]
            same = seg[: key.numel()] == seg[n - 1:]
            feats.append(key[same])
            docs.append(seg[: key.numel()][same])
        f = torch.cat(feats)
        return (f ^ (f >> 31)).remainder(length), torch.cat(docs)

    # ------------------------------------------------------------------ K8 Adam (thinc semantics)
    def adam_step(
        self,
        w: torch.Tensor,
        g: torch.Tensor,
        m1: torch.Tensor,
        m2: torch.Tensor,
        *,
        lr: float,
        beta1: float,
        beta2: float,
        eps: float,
        nr_update: int,
        grad_clip: float = 0.0,
        l2: float = 0.0,
        l2_is_weight_decay: bool = True,
        grad_scale: float = 1.0,
    ) -> None:
        """In place on fp32 ``w, m1, m2``; ``g`` is consumed (zeroed).

        g *= grad_scale; if !decoupled: g += l2*w; per-tensor clip: if ||g|| >= clip: g *= clip/||g||;
        m1 = b1*m1 + (1-b1)*g; m2 = b2*m2 + (1-b2)*g*g;
        w -= lr*sqrt(1-b2^t)/(1-b1^t) * m1/(sqrt(m2)+eps); if decoupled: w -= lr*l2*w."""
        gf = g.to(torch.float32)
        if grad_scale != 1.0:
            gf = gf * grad_scale
        if l2 != 0.0 and not l2_is_weight_decay:
            gf = gf + l2 * w
        if grad_clip and grad_clip > 0.0:
            norm = torch.linalg.vector_norm(gf)
            scale = torch.where(norm >= grad_clip, grad_clip / norm.clamp_min(1e-30), torch.ones_like(norm))
            gf = gf * scale
        fix1 = 1.0 - beta1 ** nr_update
        fix2 = 1.0 - beta2 ** nr_update
        lr_t = lr * math.sqrt(fix2) / fix1
        m1.mul_(beta1).add_(gf, alpha=1.0 - beta1)
        m2.mul_(beta2).addcmul_(gf, gf, value=1.0 - beta2)
        w.addcdiv_(m1, m2.sqrt().add_(eps), value=-lr_t)
        if l2 != 0.0 and l2_is_weight_decay:
            w.mul_(1.0 - lr * l2)
        g.zero_()

    # ------------------------------------------------------------------ misc
    def gemm(self, A: torch.Tensor, B: torch.Tensor, trans1: bool = False, trans2: bool = False) -> torch.Tensor:
        a = A.to(torch.float32)
        b = B.to(torch.float32)
        return ((a.t() if trans1 else a) @ (b.t() if trans2 else b)).to(self.dtype)

    def synchronize(self) -> None:
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)
