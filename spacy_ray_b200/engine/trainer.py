"""``Trainer``: the device-resident training step.

The generic loop (``nlp.update`` -> per-component ``update`` -> ``proxy.step``)
issues a few hundred small launches per step from Python; on a B200 that is
10x slower than the math (SURVEY.md 0.9: this workload is launch-latency bound).
``Trainer`` removes the host from the step:

* **ExampleStore** - the corpus as structure-of-arrays (attribute ids, gold
  action ids, doc offsets), built once.
* **native collate** (``native/csrc/host_runtime.cpp``) gathers the docs of a batch
  into ONE packed pinned staging buffer (padded-ragged layout + gold + per-step
  scalars), on a prefetch thread that runs while the GPU executes the previous step;
* **one H2D copy** of that buffer, issued on a side stream the moment the batch is collated
  (so it overlaps the previous step), then a device-to-device move into the static graph input;
* **one CUDA-graph replay** of the entire step - hash-embed, every tcgen05 GEMM,
  the BILUO kernel, the backward pass and the fused reduce-scatter/Adam/all-gather
  kernel - captured once per row-capacity bucket (rows rounded up to 1024);
* **one 4-byte D2H read** of the loss.

Supports any pipeline made of the built-in trainable components - a shared
``tok2vec`` plus ``tagger`` / ``ner`` / ``parser`` / ``textcat`` heads, each with its own or a
listener tok2vec (the whole of SURVEY.md 2.6's component list) - as long as the transition and
textcat heads fit their device kernels (``Trainer.unsupported_reason``).  Everything else uses the
generic ``nlp.update`` path.
"""
from __future__ import annotations

import os
import collections
import queue
import threading
import time
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence

import numpy as np
import torch

from ..models.transition_model import TransitionGold
from ..native import featurize as native
from ..nn.batch import TokenBatch
from ..nn.layers import set_dropout_rate


def _align(x: int, a: int = 256) -> int:
    return (x + a - 1) // a * a


def _kind(comp) -> Optional[str]:
    """Which device-side step serves a component.  Every token tagger (``Tagger`` and its subclasses
    ``SentenceRecognizer`` / ``Morphologizer``: same model, same kernels, only the gold ids differ) is a
    "tagger"; both document classifiers are a "textcat"."""
    from ..pipeline.components import Tagger, TextCategorizer

    if isinstance(comp, Tagger):
        return "tagger"
    if isinstance(comp, TextCategorizer):          # textcat and textcat_multilabel
        return "textcat"
    return {"Tok2VecComponent": "tok2vec", "EntityRecognizer": "ner",
            "DependencyParser": "parser"}.get(comp.__class__.__name__)


class ExampleStore:
    """Structure-of-arrays view of a list of Examples: attribute ids plus one int32 gold
    array per head.  ``slots[key] = (array, doc_off, padded)``: token-order arrays share
    ``doc_off``; *padded* arrays carry one trailing ``-1`` per doc so that a plain per-doc
    memcpy lands them in the padded-ragged row layout (the tagger's labels).  ``cats[key] = (truths,
    known)``: per-document (n_docs, n_labels) fp32 arrays of a textcat head, exactly what
    ``TextCategorizer._truths`` builds (a label missing from ``Doc.cats`` is "unknown")."""

    def __init__(self, examples: Sequence[Any], heads: Sequence[tuple]) -> None:
        lens = np.array([len(eg) for eg in examples], dtype=np.int64)
        self.doc_off = np.zeros(len(examples) + 1, dtype=np.int64)
        np.cumsum(lens, out=self.doc_off[1:])
        self.doc_off_padded = self.doc_off + np.arange(len(examples) + 1, dtype=np.int64)
        self.attrs = np.ascontiguousarray(
            np.concatenate([eg.predicted.to_array() for eg in examples]).view(np.int64))
        # dense per-column vocabulary indices: lets the collate thread group each batch's rows by
        # id with a counting sort (native.group_rows) instead of a device-side radix sort
        n_attr = self.attrs.shape[1]
        self.gid = np.empty(self.attrs.shape, dtype=np.int32)
        self.n_groups = np.zeros(n_attr, dtype=np.int32)
        for c in range(n_attr):
            uniq, inv = np.unique(self.attrs[:, c], return_inverse=True)
            self.gid[:, c] = inv.reshape(-1)
            self.n_groups[c] = len(uniq)
        self.slots: Dict[str, tuple] = {}
        self.cats: Dict[str, tuple] = {}

        def cat(parts):
            return np.ascontiguousarray(np.concatenate(parts).astype(np.int32))

        for name, comp, kind in heads:
            if kind == "ner":
                self.slots[name] = (cat([comp.gold_actions(eg.reference) for eg in examples]), self.doc_off, False)
            elif kind == "parser":
                g = [comp._gold_np(eg.reference) for eg in examples]
                self.slots[name + ".heads"] = (cat([h for h, _ in g]), self.doc_off, False)
                self.slots[name + ".labels"] = (cat([l for _, l in g]), self.doc_off, False)
            elif kind == "tagger":
                end = np.array([-1], dtype=np.int32)
                parts = []
                for eg in examples:
                    parts.append(comp.gold_ids(eg.reference).astype(np.int32))
                    parts.append(end)
                self.slots[name] = (cat(parts), self.doc_off_padded, True)
            elif kind == "textcat":
                truths, known = comp._truths(examples, "cpu")
                self.cats[name] = (np.ascontiguousarray(truths.numpy()), np.ascontiguousarray(known.numpy()))
        self.lens = lens
        self.n_docs = len(examples)
        self.max_len = int(lens.max()) if len(lens) else 1


@dataclass
class _Layout:
    rows: int
    docs: int
    lmax: int
    slots: tuple = ()
    cats: tuple = ()                 # ((textcat head, n_labels), ...)
    bucket: int = 1024
    n_attr: int = 4
    off_attrs: int = 0
    off_mask: int = 0
    off_starts: int = 0
    off_lens: int = 0
    off_tok: int = 0
    off_gold: Any = None
    off_inv: int = 0
    off_meta: int = 0
    nbytes: int = 0

    def __post_init__(self):
        o = 0
        self.off_attrs = o; o = _align(o + self.rows * 4 * 8)
        self.off_mask = o; o = _align(o + self.rows * 4)
        self.off_starts = o; o = _align(o + self.docs * 4)
        self.off_lens = o; o = _align(o + self.docs * 4)
        self.off_tok = o; o = _align(o + self.docs * 4)
        self.off_gold = {}
        for key in self.slots:
            self.off_gold[key] = o; o = _align(o + self.rows * 4)
        self.off_cats = {}
        for key, n_labels in self.cats:
            off_t = o; o = _align(o + self.docs * n_labels * 4)
            self.off_cats[key] = (off_t, o, n_labels); o = _align(o + self.docs * n_labels * 4)
        self.off_scratch = o; o = _align(o + self.docs * 4)
        self.off_perm = o; o = _align(o + self.n_attr * self.rows * 4)
        self.off_inv = o; o = _align(o + self.lmax * 4)
        self.off_meta = o; o = _align(o + 16)
        self.nbytes = o


class _Views:
    """Typed views into one packed byte buffer (host numpy or device torch)."""

    def __init__(self, lay: _Layout, buf: torch.Tensor):
        self.buf = buf

        def v(off, n, dt):
            return buf[off: off + n * torch.tensor([], dtype=dt).element_size()].view(dt)

        self.attrs = v(lay.off_attrs, lay.rows * 4, torch.int64).view(lay.rows, 4)
        self.mask = v(lay.off_mask, lay.rows, torch.float32)
        self.starts = v(lay.off_starts, lay.docs, torch.int32)
        self.lens = v(lay.off_lens, lay.docs, torch.int32)
        self.tok_off = v(lay.off_tok, lay.docs, torch.int32)
        self.gold = {k: v(off, lay.rows, torch.int32) for k, off in lay.off_gold.items()}
        self.cats = {k: tuple(v(off, lay.docs * n, torch.float32).view(lay.docs, n) for off in (ot, ok))
                     for k, (ot, ok, n) in lay.off_cats.items()}     # textcat (truths, known)
        self.scratch = v(lay.off_scratch, lay.docs, torch.int32)
        self.perm = v(lay.off_perm, lay.n_attr * lay.rows, torch.int32)
        self.inv_active = v(lay.off_inv, lay.lmax, torch.float32)
        self.meta = v(lay.off_meta, 4, torch.int32)


def make_stage(lay: _Layout, store: ExampleStore, pin: bool = True) -> dict:
    """One packed host staging buffer (pinned for the async H2D copy) + numpy views into it."""
    hb = torch.zeros(lay.nbytes, dtype=torch.uint8, pin_memory=pin)
    hv = _Views(lay, hb)
    arrs = {k: getattr(hv, k).numpy() for k in
            ("attrs", "mask", "starts", "lens", "tok_off", "inv_active", "meta", "scratch", "perm")}
    arrs["gold"] = {k: t.numpy() for k, t in hv.gold.items()}
    arrs["cats"] = {k: (t.numpy(), kn.numpy()) for k, (t, kn) in hv.cats.items()}
    arrs["hist"] = np.zeros(int(store.n_groups.sum()) + len(store.n_groups), dtype=np.int32)
    for key, (_arr, _off, padded) in store.slots.items():
        if padded:
            arrs["gold"][key][:] = -1              # rows past the batch carry "no gold"
    return {"buf": hb, "np": arrs, "event": None, "rows": 0, "docs": 0, "words": 0}


def fill_stage(st: ExampleStore, lay: _Layout, stage: dict, ids: np.ndarray, hist: Optional[np.ndarray] = None) -> None:
    """Gather docs ``ids`` into the packed staging buffer (native memcpy loops).  ``hist``: counting-sort
    scratch sized for ``st``'s vocabulary (default: the stage's own, sized for the trainer's store)."""
    if stage["event"] is not None:
        stage["event"].synchronize()               # previous H2D out of this buffer has completed
    a = stage["np"]
    ids = np.ascontiguousarray(ids, dtype=np.int64)
    rows = native.collate(st.attrs, st.doc_off, ids, a["attrs"], a["mask"], a["starts"], a["lens"])
    words = int(st.lens[ids].sum())
    first = True
    for key, (arr, doc_off, padded) in st.slots.items():
        out = a["gold"][key]
        if padded:                                 # row 0 is the batch's leading pad row
            out[0] = -1
            used = native.collate_gold(arr, doc_off, ids, out[1:], a["scratch"])
            out[1 + used: max(stage["rows"], 1 + used)] = -1
        else:
            native.collate_gold(arr, doc_off, ids, out, a["tok_off"] if first else a["scratch"])
            first = False
    n = len(ids)
    for key, (truths, known) in st.cats.items():   # per-doc textcat truths: one vectorised gather
        out_t, out_k = a["cats"][key]
        np.take(truths, ids, axis=0, out=out_t[:n])
        np.take(known, ids, axis=0, out=out_k[:n])
        out_t[n:] = 0.0
        out_k[n:] = 0.0                            # unused doc slots: nothing known
    if first:                                      # no token-order slot filled tok_off
        lens_i = st.lens[ids]
        a["tok_off"][: len(ids)] = (np.cumsum(lens_i) - lens_i).astype(np.int32)
    if len(ids) < lay.docs:                        # partial batch: the unused doc slots are empty docs
        a["lens"][len(ids):] = 0
        a["starts"][len(ids):] = 0
        a["tok_off"][len(ids):] = 0
    lens = a["lens"][: len(ids)]
    counts = (lens[None, :] > np.arange(lay.lmax, dtype=np.int32)[:, None]).sum(axis=1)
    a["inv_active"][:] = 1.0 / np.maximum(counts, 1)
    a["meta"][0] = rows
    a["meta"][1] = len(ids)                        # real doc count (textcat: loss and gradient scale)
    # HashEmbed backward: rows grouped by id per attribute column, laid out for the row bucket
    # the step will run with (the captured graph reads perm as (n_attr, rb))
    rb = min(lay.rows, _align(int(rows), lay.bucket))
    native.group_rows(st.gid, st.n_groups, st.doc_off, ids, rb, a["perm"], a["hist"] if hist is None else hist)
    stage["rows"], stage["docs"], stage["words"] = int(rows), len(ids), int(words)


class Trainer:
    @staticmethod
    def unsupported_reason(nlp, max_len: Optional[int] = None) -> Optional[str]:
        """Why this pipeline cannot run device-resident (None = it can)."""
        heads = [(n, c, _kind(c)) for n, c in nlp.pipeline if getattr(c, "is_trainable", False)]
        if not heads:
            return "no trainable component"
        for name, comp, kind in heads:
            if kind is None:
                return f"component {name!r} ({comp.__class__.__name__}) has no device-side update"
            if any(node.name == "staticvectors" for node in comp.model.walk()):
                return f"{name}: static vectors (row lookup is host-side; generic path)"
            if kind in ("ner", "parser"):
                lower = comp.model.get_ref("lower").get_param("W")
                _nF, nO, nP, _nI = lower.shape
                nA = comp.system.n_actions
                if kind == "ner" and (nP != 2 or nO % 32 or (nO * nP) // 32 > 8 or nA > 256):
                    return f"{name}: hidden_width/maxout_pieces outside the BILUO kernel's range"
                if kind == "parser" and (nO % 32 or nO // 32 not in (1, 2, 4) or nP not in (2, 3) or nA > 192):
                    return f"{name}: hidden_width/maxout_pieces/labels outside the arc-eager kernel's range"
                if kind == "parser" and max_len is not None:
                    cap = Trainer.parser_doc_capacity(comp)
                    if max_len > cap:
                        return f"{name}: documents longer than {cap} tokens"
            if kind == "textcat":
                why = Trainer.textcat_reason(comp)
                if why is not None:
                    return f"{name}: {why}"
        if all(kind == "tok2vec" for _, _, kind in heads):
            return "no head component"
        return None

    @staticmethod
    def textcat_reason(comp) -> Optional[str]:
        """Why the textcat kernels cannot serve this head (None = they can): label count, pooled width
        (n_pool * width) and n-gram size must fit what one CTA per document holds."""
        from ..ops.b200_ops import TEXTCAT_MAX_LABELS, TEXTCAT_MAX_NGRAM, TEXTCAT_MAX_POOL

        model = comp.model
        if "update_with_cats" not in model.attrs:
            return f"model {model.name!r} has no device-side update"
        n_labels = len(comp.labels) or model.maybe_get_dim("nO") or 0
        if n_labels > TEXTCAT_MAX_LABELS:
            return f"{n_labels} labels (the textcat kernels hold at most {TEXTCAT_MAX_LABELS})"
        if model.has_ref("output"):
            pool = model.get_ref("output").maybe_get_dim("nI") or 0
            if pool > TEXTCAT_MAX_POOL:
                return f"pooled width {pool} (n_pool * width; the textcat kernels hold at most {TEXTCAT_MAX_POOL})"
        bow = model.get_ref("linear_model") if model.has_ref("linear_model") else (
            model if model.name == "textcat_bow" else None)
        if bow is not None:
            n = int(bow.attrs.get("ngram_size", 1))
            if not 1 <= n <= TEXTCAT_MAX_NGRAM:
                return f"ngram_size {n} (the textcat kernels hash 1 to {TEXTCAT_MAX_NGRAM})"
        return None

    @staticmethod
    def parser_doc_capacity(comp) -> int:
        """Longest doc the device arc-eager kernel can hold for this parser head (its per-warp state
        lives in shared memory next to the staged upper-layer weights)."""
        ops = comp.model.ops
        fn = getattr(ops, "arc_eager_capacity", None)
        if fn is None:
            return 128
        _nF, nO, nP, _nI = comp.model.get_ref("lower").get_param("W").shape
        return int(fn(int(nO), int(nP), int(comp.system.n_actions)))

    def __init__(self, nlp, proxy, examples: Sequence[Any], *, docs_per_batch: int, dropout: float = 0.1,
                 component: Optional[str] = None, use_graphs: bool = True, bucket_rows: int = 256,
                 prefetch: bool = True, n_stage: int = 3, exchange: bool = True, prefetch_workers: int = 2):
        self.nlp, self.proxy = nlp, proxy
        # exchange=False: the captured step only ACCUMULATES gradients (accumulate_gradient > 1: the caller
        # runs proxy.step() once per full batch, after the last micro-batch)
        self.exchange = bool(exchange)
        self.heads = [(n, c, _kind(c)) for n, c in nlp.pipeline if getattr(c, "is_trainable", False)]
        self.loss_names = [n for n, _c, k in self.heads if k != "tok2vec"]
        self.ops = self.heads[0][1].model.ops
        if self.ops.device.type != "cuda":
            raise ValueError("Trainer needs the CUDA backend; use nlp.update on CPU")
        self.device = self.ops.device
        self.dropout = float(dropout)
        self.B = int(docs_per_batch)
        self.store = ExampleStore(examples, self.heads)
        # the arc-eager kernel keeps a document's state in shared memory (several hundred tokens fit):
        # longer documents stay in the store but batches containing one are handed back to the generic path
        caps = [self.parser_doc_capacity(c) for _n, c, k in self.heads if k == "parser"]
        self.max_doc_len = min(caps) if caps else None
        cap_len = self.store.max_len if self.max_doc_len is None else min(self.store.max_len, self.max_doc_len)
        why = self.unsupported_reason(nlp, cap_len)
        if why is not None:
            raise ValueError(f"pipeline not supported by the device-resident engine: {why}")
        self._doc_index = {id(eg.reference): i for i, eg in enumerate(examples)}
        self.bucket_rows = int(bucket_rows)
        rows_cap = _align(self.B * cap_len + self.B + 1, self.bucket_rows)
        self.lay = _Layout(rows=rows_cap, docs=self.B, lmax=_align(cap_len, 64),
                           slots=tuple(self.store.slots), bucket=self.bucket_rows,
                           cats=tuple((k, int(t.shape[1])) for k, (t, _kn) in self.store.cats.items()),
                           n_attr=int(self.store.attrs.shape[1]))
        if hasattr(self.ops, "max_rows_hint"):
            self.ops.max_rows_hint = max(int(self.ops.max_rows_hint), int(rows_cap))
        self.host_grouping = os.environ.get("SRB_HOST_GROUP", "1") != "0"
        self.head_streams = os.environ.get("SRB_HEAD_STREAMS", "1") != "0"
        self._head_streams: List[torch.cuda.Stream] = []
        self.use_graphs = use_graphs
        self.dev_buf = torch.zeros(self.lay.nbytes, dtype=torch.uint8, device=self.device)
        self.dv = _Views(self.lay, self.dev_buf)
        n_stage = max(int(n_stage), (int(prefetch_workers) if prefetch else 1) + 2)
        self.stages = [make_stage(self.lay, self.store, pin=True) for _ in range(n_stage)]
        for stage in self.stages:
            # device landing buffer of this stage: the H2D copy runs on a side stream as soon as the
            # batch is collated (i.e. while the previous step still executes); the step itself
            # only does a device-to-device copy into the static graph input
            stage["land"] = torch.zeros(self.lay.nbytes, dtype=torch.uint8, device=self.device)
            stage["consumed"] = None
        self._loss_slots = [{"buf": torch.zeros(max(8, len(self.loss_names)), dtype=torch.float32, pin_memory=True),
                             "ev": torch.cuda.Event(),
                             "n": 0} for _ in range(2)]
        self._pending_loss: Optional[dict] = None
        self._graphs: Dict[int, Any] = {}
        self._pool = torch.cuda.graph_pool_handle() if use_graphs else None
        self._warmed = False
        self._loss_out: Dict[int, torch.Tensor] = {}
        self._launches_per_replay: Dict[int, int] = {}
        self.h2d_bytes_per_step = self.lay.nbytes
        self.steps = 0
        self.adhoc_batches = 0               # batches collated from a throw-away store (docs not in the store)
        self._stage_i = 0
        self._prefetch = prefetch
        self._q_in: "queue.Queue" = queue.Queue()
        # batches prepared but not yet consumed, in submission order (several collate workers may
        # finish out of order; ``_take`` hands them out in the order ``prepare`` was called)
        self._pending: "collections.deque" = collections.deque()
        self._threads: List[threading.Thread] = []
        # How many batches a caller should keep prepared ahead of the step it is about to run.  Starts at
        # 1 (one collate in flight is enough when the device step is longer than a collate, and a second
        # busy worker costs the launching thread ~2 % through the GIL / driver lock: flagship 99 % -> 97 %
        # of device-timed); ``_take`` raises it to the number of workers when one collate costs more than
        # half the period at which batches are consumed (tagger w96: 0.33 ms step, collate about as long:
        # 82 % -> 96 % of device-timed).
        self._workers = max(1, min(int(prefetch_workers), len(self.stages) - 2)) if prefetch else 1
        self.prefetch_depth = 1
        self._takes = 0
        self._period = 0.0
        self._cost = 0.0
        self._last_take: Optional[float] = None
        self._side = torch.cuda.Stream(device=self.device)
        # the captured step runs at high stream priority: the backend's side-stream work (weight-
        # gradient GEMMs, default priority) then only takes SMs the dependent chain leaves idle
        self._hp = torch.cuda.Stream(device=self.device, priority=-1)
        if prefetch:
            # collation is native code called through ctypes (the GIL is released): two workers give
            # two batches in flight, which the 0.33 ms tagger step needs (one collate takes about as long)
            for _ in range(self._workers):
                t = threading.Thread(target=self._prefetch_loop, daemon=True)
                t.start()
                self._threads.append(t)

    # ------------------------------------------------------------------ host side
    def _fill(self, stage: dict, ids: np.ndarray) -> None:
        fill_stage(self.store, self.lay, stage, ids)

    def _upload(self, stage: dict) -> None:
        """Async H2D of a filled staging buffer into its landing buffer, on the side stream."""
        with torch.cuda.stream(self._side):
            if stage["consumed"] is not None:
                self._side.wait_event(stage["consumed"])   # the step that read this landing buffer is done with it
            stage["land"].copy_(stage["buf"], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._side)
        stage["event"] = ev

    def _produce(self, ticket: dict) -> None:
        stage = ticket["stage"]
        try:
            ev = stage.get("event")
            if ev is not None:
                ev.synchronize()                # the previous H2D copy out of this pinned buffer has finished
            t0 = time.perf_counter()
            self._fill(stage, ticket["ids"])
            self._upload(stage)
            ticket["cost"] = time.perf_counter() - t0
        except BaseException as e:              # surfaced in the training thread by _take()
            ticket["err"] = e
        ticket["done"].set()

    def _prefetch_loop(self) -> None:
        torch.cuda.set_device(self.device)
        while True:
            ticket = self._q_in.get()
            if ticket is None:
                return
            self._produce(ticket)

    def prepare(self, ids: np.ndarray) -> None:
        """Queue the collation of a future batch (returns immediately).  Up to ``prefetch_depth``
        batches may be prepared ahead of the step that is about to run."""
        if self.max_doc_len is not None and len(ids) and int(self.store.lens[ids].max()) > self.max_doc_len:
            raise ValueError(f"batch contains a document longer than {self.max_doc_len} tokens; "
                             "use nlp.update (generic path) for it")
        if len(self._pending) >= len(self.stages) - 1:
            raise RuntimeError(f"{len(self._pending)} batches prepared and not consumed: the staging ring has "
                               f"{len(self.stages)} buffers (prepare at most prefetch_depth = {self.prefetch_depth} ahead)")
        stage = self.stages[self._stage_i]
        self._stage_i = (self._stage_i + 1) % len(self.stages)
        ticket = {"stage": stage, "ids": ids, "done": threading.Event(), "err": None}
        self._pending.append(ticket)
        if self._prefetch:
            self._q_in.put(ticket)
        else:
            self._produce(ticket)

    def _take(self) -> dict:
        """The oldest prepared batch (its staging record), in the order ``prepare`` was called."""
        ticket = self._pending.popleft()
        ticket["done"].wait()
        if self.prefetch_depth < self._workers:
            # host-bound?  compare what a collate costs with the period at which batches are consumed
            now = time.perf_counter()
            if self._last_take is not None:
                self._takes += 1
                self._period += now - self._last_take
                self._cost += ticket.get("cost", 0.0)
                if self._takes >= 8:
                    if self._cost > 0.5 * self._period:
                        self.prefetch_depth = self._workers
                    self._takes, self._period, self._cost = 0, 0.0, 0.0
            self._last_take = now
        if ticket["err"] is not None:
            raise ticket["err"]
        return ticket["stage"]

    # ------------------------------------------------------------------ device side
    def _batch_views(self, rows: int) -> tuple:
        dv = self.dv
        tb = TokenBatch(
            attrs=dv.attrs[:rows], mask=dv.mask[:rows].view(rows, 1), doc_starts=dv.starts, doc_lens=dv.lens,
            lengths=[], starts=[], n_tokens=rows, n_rows=rows,
        )
        tb.extra["tok_off"] = dv.tok_off
        tb.extra["inv_active"] = dv.inv_active
        tb.extra["max_len"] = int(self.lay.lmax)
        if self.host_grouping:
            n_attr = self.lay.n_attr
            tb.extra["embed_perm"] = dv.perm[: n_attr * rows].view(n_attr, rows)
        return tb

    def _step_fn(self, rows: int) -> torch.Tensor:
        """Forward + backward of every component, then the gradient exchange + optimizer.
        Returns the per-head losses as one small device vector (``loss_names`` order)."""
        tb = self._batch_views(rows)
        gold = self.dv.gold
        stamp = getattr(self.proxy.comm, "stamp", None)
        if stamp is not None:
            stamp(0)                                        # trace: step start
        if self.exchange and hasattr(self.proxy, "begin_step"):
            self.proxy.begin_step(overlap=True)             # buckets are exchanged under the backward pass
        bump = getattr(getattr(self.ops, "k", None), "bump_i64", None)
        if bump is not None and self.ops.seed_dev.is_cuda:
            bump(self.ops.seed_dev, 7919)                   # fresh dropout masks on every replay (1-thread kernel)
        else:
            self.ops.seed_dev.add_(7919)
        shared = [c for _n, c, k in self.heads if k == "tok2vec"]
        n_heads = sum(1 for _n, _c, k in self.heads if k != "tok2vec")
        # heads that listen to ONE shared tok2vec are independent of each other: run each on its own
        # stream (the transition kernels occupy ~7 % of the SMs), then sum their gradients and run
        # the tok2vec backward once on the main stream
        concurrent = self.head_streams and len(shared) == 1 and n_heads >= 2
        main = torch.cuda.current_stream(self.device)
        forked = []
        losses = []
        for name, comp, kind in self.heads:
            if kind == "tok2vec":
                # forward now; its backward fires when the last listener returns its gradient
                comp.update((), batch=tb, drop=self.dropout, sgd=False, losses=None, defer_backprop=concurrent)
                continue
            stream = main
            if concurrent:
                stream = self._head_stream(len(forked))
                stream.wait_stream(main)
                forked.append(stream)
            with torch.cuda.stream(stream):
                set_dropout_rate(comp.model, self.dropout)
                if kind == "tagger":
                    loss, _ = comp.model.attrs["update_with_labels"](tb, gold[name][:rows].to(torch.int64))
                elif kind == "textcat":
                    truths, known = self.dv.cats[name]
                    loss, _ = comp.model.attrs["update_with_cats"](tb, truths, known, self.dv.meta[1:2])
                elif kind == "ner":
                    g = TransitionGold(actions=gold[name][:rows], offsets=None)
                    loss = comp.model.attrs["run"](tb, comp.system, g, True).loss
                else:
                    g = TransitionGold(heads_flat=gold[name + ".heads"][:rows], labels_flat=gold[name + ".labels"][:rows])
                    loss = comp.model.attrs["run"](tb, comp.system, g, True).loss
                losses.append(loss.reshape(()).to(torch.float32))
        if concurrent:
            for stream in forked:
                main.wait_stream(stream)
            shared[0].finish_backprop()
        if stamp is not None:
            stamp(1)                                        # trace: forward + backward enqueued, before the final join
        if self.exchange:
            self.proxy.step()
        else:
            join = getattr(self.ops, "join_side", None)
            if join is not None:
                join()                                      # side-stream weight-gradient GEMMs rejoin the capture stream
        if stamp is not None:
            stamp(2)                                        # trace: exchange joined = step end
        return losses[0].reshape(1) if len(losses) == 1 else torch.stack(losses)

    def _head_stream(self, i: int) -> "torch.cuda.Stream":
        while len(self._head_streams) <= i:
            self._head_streams.append(torch.cuda.Stream(device=self.device, priority=-1))
        return self._head_streams[i]

    def _bucket(self, rows: int) -> int:
        return min(self.lay.rows, _align(rows, self.bucket_rows))

    def _run(self, rows: int) -> torch.Tensor:
        rb = self._bucket(rows)
        comm = self.proxy.comm
        if not self.use_graphs or not self._warmed:
            # The very first step runs eagerly on every rank (in lockstep): it performs the
            # one-time kernel attribute setup / workspace allocation that must not happen
            # under capture, and it is a real training step.
            self._warmed = True
            return self._step_fn(rb)
        g = self._graphs.get(rb)
        if g is None:
            g = self._capture(rb)
        if hasattr(comm, "_sync_hyper"):
            comm._sync_hyper()                 # learning-rate schedules: the kernel reads the device copy
        g.replay()
        if self.exchange and hasattr(comm, "host_bookkeeping"):
            comm.host_bookkeeping()
        n_ops, n_comm = self._launches_per_replay[rb]
        self.ops.launches += n_ops
        if hasattr(comm, "launches"):
            comm.launches += n_comm
        return self._loss_out[rb]

    def _capture(self, rb: int):
        """Capture the whole step for row-capacity ``rb``.  Capturing executes nothing, so
        ranks may capture different buckets at different times without unbalancing the
        collective inside the step; all buckets share one memory pool."""
        comm = self.proxy.comm
        if hasattr(comm, "_sync_hyper"):
            comm._sync_hyper()
        if hasattr(comm, "reset_gates"):
            comm.reset_gates()                 # the first consumer of every bucket carries its gate in the graph
        torch.cuda.synchronize(self.device)
        l0, c0 = self.ops.launches, getattr(comm, "launches", 0)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, pool=self._pool, stream=self._hp):
            loss = self._step_fn(rb)
        self._launches_per_replay[rb] = (self.ops.launches - l0, getattr(comm, "launches", 0) - c0)
        self.ops.launches = l0
        if hasattr(comm, "launches"):
            comm.launches = c0
        self._graphs[rb] = g
        self._loss_out[rb] = loss
        return g

    def rows_for(self, ids: np.ndarray) -> int:
        return int(self.store.lens[ids].sum()) + len(ids) + 1

    def capture_buckets(self, rows_list: Sequence[int]) -> List[int]:
        """Pre-capture the graphs for the given row counts (after the first eager step)."""
        if not self.use_graphs or not self._warmed:
            return []
        done = []
        for rb in sorted({self._bucket(r) for r in rows_list}):
            if rb not in self._graphs:
                self._capture(rb)
                done.append(rb)
        return done

    def step_async(self) -> torch.Tensor:
        """Consume the next prepared batch: H2D copy + (graph) step.  Returns the loss tensor
        (device); reading it is the caller's D2H sync."""
        stage = self._take()
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(stage["event"])                              # the packed H2D copy (side stream)
        self.dev_buf.copy_(stage["land"], non_blocking=True)        # D2D into the static graph input
        done = torch.cuda.Event()
        done.record(cur)
        stage["consumed"] = done
        loss = self._run(stage["rows"])
        self.steps += 1
        self.last = {"docs": stage["docs"], "words": stage["words"], "rows": stage["rows"]}
        return loss

    def train_step(self, ids: Optional[np.ndarray] = None, *, lag: int = 1) -> float:
        """The public one-call step: (collate if ``ids`` given) -> H2D -> step -> loss (D2H).

        Every step's per-head losses are copied to pinned host memory right behind the step
        (async D2H on the step's stream).  With ``lag=1`` (default) the call returns the loss of
        the PREVIOUS step - whose copy has long finished - so the host never stalls the device
        between steps (the first call returns its own loss); ``lag=0`` blocks on this step.
        ``flush_loss()`` returns the one still in flight."""
        if ids is not None:
            self.prepare(ids)
        loss = self.step_async()
        slot = self._loss_slots[self.steps % len(self._loss_slots)]
        slot["buf"][: loss.numel()].copy_(loss, non_blocking=True)
        slot["n"] = int(loss.numel())
        slot["ev"].record()
        if lag <= 0:
            prev, self._pending_loss = slot, None
        else:
            prev, self._pending_loss = self._pending_loss, slot
            if prev is None:                           # first call: nothing older to report
                prev = slot
        prev["ev"].synchronize()
        return float(prev["buf"][: prev["n"]].sum())

    def flush_loss(self) -> Optional[float]:
        """Loss of the most recent step (blocks until it has been computed)."""
        slot = self._pending_loss
        if slot is None:
            return None
        slot["ev"].synchronize()
        return float(slot["buf"][: slot["n"]].sum())

    def losses_dict(self, loss_vec: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {n: loss_vec[i] for i, n in enumerate(self.loss_names)}

    def ids_for(self, examples: Sequence[Any]) -> Optional[np.ndarray]:
        """Store indices of ``examples`` (matched by the identity of their reference Doc), or
        None if any of them is not part of the store / the batch exceeds the staging capacity."""
        if len(examples) > self.B:
            return None
        idx = self._doc_index
        out = np.empty(len(examples), dtype=np.int64)
        for i, eg in enumerate(examples):
            j = idx.get(id(eg.reference))
            if j is None:
                return None
            out[i] = j
        if self.rows_for(out) > self.lay.rows:
            return None
        if self.max_doc_len is not None and int(self.store.lens[out].max(initial=0)) > self.max_doc_len:
            return None
        return out

    def update_examples(self, examples: Sequence[Any]) -> Optional[torch.Tensor]:
        """``nlp.update`` fast path: returns the loss tensor (no host sync), or None when the batch does
        not fit the staging capacity (the caller then takes the generic path).  Batches whose docs are
        not in the store - a streamed corpus (``max_epochs = -1``), a corpus too large to pre-load - are
        collated through a throw-away store built from the batch itself."""
        ids = self.ids_for(examples)
        if ids is not None:
            self.prepare(ids)
            return self.step_async()
        if len(examples) > self.B:
            return None
        lens = [len(eg) for eg in examples]
        if not lens or sum(lens) + len(lens) + 1 > self.lay.rows or max(lens) > self.lay.lmax:
            return None
        if self.max_doc_len is not None and max(lens) > self.max_doc_len:
            return None
        adhoc = ExampleStore(examples, self.heads)
        stage = self.stages[self._stage_i]
        self._stage_i = (self._stage_i + 1) % len(self.stages)
        hist = np.zeros(int(adhoc.n_groups.sum()) + len(adhoc.n_groups), dtype=np.int32)
        ev = stage.get("event")
        if ev is not None:
            ev.synchronize()
        fill_stage(adhoc, self.lay, stage, np.arange(len(examples), dtype=np.int64), hist=hist)
        self._upload(stage)
        done = threading.Event()
        done.set()
        self._pending.append({"stage": stage, "ids": None, "done": done, "err": None})
        self.adhoc_batches += 1
        return self.step_async()

    def batches(self, n: int, seed: int = 0, tokens_per_batch: Optional[int] = None) -> List[np.ndarray]:
        """``n`` random batches of ``B`` docs.  With ``tokens_per_batch`` every batch is adjusted (a few
        docs swapped for longer / shorter ones) to hold exactly that many tokens: data-parallel ranks
        then run the same row count every step - a synchronous step is as slow as its largest batch,
        so random-length batches cost ~sigma/mean of throughput at 8 ranks - and one CUDA graph serves
        every step (the spaCy default batcher, ``batch_by_words``, equalises words for the same reason)."""
        rng = np.random.default_rng(seed)
        out = []
        perm = rng.permutation(self.store.n_docs)
        pos = 0
        lens = self.store.lens
        by_len: Dict[int, np.ndarray] = {}
        if tokens_per_batch is not None:
            for L in np.unique(lens):
                by_len[int(L)] = np.nonzero(lens == L)[0]
            lo, hi = int(lens.min()), int(lens.max())
        for _ in range(n):
            if pos + self.B > len(perm):
                perm = rng.permutation(self.store.n_docs)
                pos = 0
            ids = perm[pos:pos + self.B].astype(np.int64)
            pos += self.B
            if tokens_per_batch is not None:
                diff = int(tokens_per_batch) - int(lens[ids].sum())
                tries = 0
                while diff != 0 and tries < 64 * self.B:
                    tries += 1
                    i = int(rng.integers(len(ids)))
                    want = int(np.clip(int(lens[ids[i]]) + diff, lo, hi))
                    cand = by_len.get(want)
                    if cand is None or want == int(lens[ids[i]]):
                        continue
                    diff -= want - int(lens[ids[i]])
                    ids[i] = int(cand[rng.integers(len(cand))])
                if diff != 0:
                    raise ValueError(f"could not balance a batch to {tokens_per_batch} tokens (off by {diff})")
            out.append(np.sort(ids).astype(np.int64))
        return out

    def close(self) -> None:
        for _ in self._threads:
            self._q_in.put(None)
        for t in self._threads:
            t.join(timeout=5)
        self._threads = []
