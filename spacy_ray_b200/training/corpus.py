"""Corpus readers.

``spacy.Corpus.v1`` reads what upstream reads - binary ``.spacy`` DocBin files
(``training/docbin.py`` implements the container without spaCy; the reference's
``bin/get-data.sh:6-13`` produces them with ``spacy convert``) - and, in the same
directory walk, JSON-lines files (one doc per line: ``{"words", "tags", "ents",
"heads", "deps"}`` or Prodigy-style ``{"text", "spans"}``, the raw format that script
downloads).  An empty/None path yields nothing, which is what the reference's only
test relies on (``spacy_ray/tests/test_worker.py:26-29``).

``spacy_ray_b200.SyntheticCorpus.v1`` generates a seeded, *learnable* synthetic
corpus (there is no network for real data): Zipfian vocabulary, per-type tags,
capitalised multi-word entities, projective dependency trees, and document
categories (``textcat``: one of two exclusive classes; ``textcat_multilabel``: two
independent ones) that follow from which marker words a doc contains.
"""
from __future__ import annotations

import json
from pathlib import Path
from typing import Any, Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np

from ..config import registry
from ..pipeline.doc import Doc, Example, featurize_words


class JsonlCorpus:
    def __init__(self, path: Optional[str], *, max_length: int = 0, limit: int = 0, gold_preproc: bool = False,
                 augmenter: Any = None, shuffle: bool = False):
        self.path = Path(path) if path else None
        self.max_length = max_length
        self.limit = limit
        self._cache: Optional[List[Doc]] = None

    def _files(self) -> List[Path]:
        if self.path is None or str(self.path) in ("", "."):
            return []
        if self.path.is_dir():
            return sorted(p for p in self.path.rglob("*") if p.suffix in (".jsonl", ".json", ".spacy"))
        if not self.path.exists():
            raise FileNotFoundError(f"Corpus path not found: {self.path}")
        return [self.path]

    def _load(self) -> List[Doc]:
        if self._cache is None:
            docs: List[Doc] = []
            for f in self._files():
                if self.limit and len(docs) >= self.limit:
                    break
                if f.suffix == ".spacy":
                    from .docbin import DocBin

                    for d in DocBin().from_disk(f).get_docs():
                        if len(d) == 0 or (self.max_length and len(d) > self.max_length):
                            continue
                        docs.append(d)
                        if self.limit and len(docs) >= self.limit:
                            break
                    continue
                with f.open("r", encoding="utf8") as fh:
                    for line in fh:
                        line = line.strip()
                        if not line:
                            continue
                        d = Doc.from_dict(json.loads(line))
                        if len(d) == 0 or (self.max_length and len(d) > self.max_length):
                            continue
                        docs.append(d)
                        if self.limit and len(docs) >= self.limit:
                            break
            self._cache = docs
        return self._cache

    def __call__(self, nlp=None) -> Iterator[Example]:
        for doc in self._load():
            yield Example.from_doc(doc)


@registry.readers("spacy.Corpus.v1")
def create_docbin_reader(path: Optional[str] = None, gold_preproc: bool = False, max_length: int = 0,
                         limit: int = 0, augmenter: Any = None) -> JsonlCorpus:
    return JsonlCorpus(path, max_length=max_length, limit=limit, gold_preproc=gold_preproc, augmenter=augmenter)


@registry.readers("spacy.JsonlCorpus.v1")
def create_jsonl_reader(path: Optional[str] = None, min_length: int = 0, max_length: int = 0, limit: int = 0) -> JsonlCorpus:
    return JsonlCorpus(path, max_length=max_length, limit=limit)


# ----------------------------------------------------------------------------
_SYL = ["ka", "to", "mi", "ne", "ra", "su", "lo", "vi", "de", "pa", "no", "ti", "se", "mu", "ro", "li",
        "ba", "ko", "fe", "gu", "za", "xi", "yo", "wu", "qe", "ha", "jo", "pe", "ni", "ta", "sa", "me"]
TAGS = ["NOUN", "VERB", "ADJ", "ADV", "DET", "ADP", "PRON", "PROPN", "NUM", "PUNCT", "CCONJ", "AUX",
        "PART", "SCONJ", "INTJ", "SYM", "X"]
ENT_LABELS = ["PERSON", "ORG", "GPE", "LOC", "PRODUCT", "EVENT", "DATE", "TIME", "MONEY", "PERCENT",
              "FAC", "NORP", "LAW", "LANGUAGE", "WORK_OF_ART", "QUANTITY", "ORDINAL", "CARDINAL"]
DEP_LABELS = ["nsubj", "obj", "det", "amod", "advmod", "case", "nmod", "obl", "cc", "conj", "aux",
              "mark", "compound", "punct", "nummod", "appos"]
# document categories: a doc "has" a marker when it contains that vocabulary entry.  Entries 2 and 3 of the
# Zipfian vocabulary occur in roughly half / a third of 24-token docs.
CAT_MARKERS = (2, 3)


def doc_cats(ids: np.ndarray, multilabel: bool) -> Dict[str, float]:
    """The categories of a doc with vocabulary ids ``ids``: a function of its content alone (no random
    draw, so adding a textcat task leaves every other annotation of the corpus unchanged)."""
    has = [bool(np.any(ids == m)) for m in CAT_MARKERS]
    if multilabel:
        return {"MARK_A": float(has[0]), "MARK_B": float(has[1])}
    return {"MARKED": float(has[0]), "PLAIN": float(not has[0])}


def _make_word(i: int, rng: np.random.Generator) -> str:
    n = 1 + (i % 3) + int(rng.integers(0, 2))
    return "".join(_SYL[int(rng.integers(0, len(_SYL)))] for _ in range(n))


class SyntheticCorpus:
    """Deterministic synthetic corpus.  ``tasks`` selects which gold layers are
    produced.  All docs are generated (and featurised) once, on first use."""

    def __init__(self, n_docs: int = 2000, seed: int = 0, min_len: int = 8, max_len: int = 40,
                 vocab_size: int = 20000, n_tags: int = 17, n_ent_labels: int = 4, n_dep_labels: int = 8,
                 ent_rate: float = 0.12, noise: float = 0.02, tasks: Sequence[str] = ("tagger", "ner", "parser"),
                 vocab_seed: int = 0):
        self.n_docs, self.seed = int(n_docs), int(seed)
        self.vocab_seed = int(vocab_seed)       # shared by train/dev corpora so word types (and their tags) agree
        self.min_len, self.max_len = int(min_len), int(max_len)
        self.vocab_size = int(vocab_size)
        self.n_tags = min(int(n_tags), len(TAGS))
        self.n_ent_labels = min(int(n_ent_labels), len(ENT_LABELS))
        self.n_dep_labels = min(int(n_dep_labels), len(DEP_LABELS))
        self.ent_rate, self.noise = float(ent_rate), float(noise)
        self.tasks = tuple(tasks)
        if "textcat" in self.tasks and "textcat_multilabel" in self.tasks:
            raise ValueError("SyntheticCorpus: choose one of the tasks 'textcat' / 'textcat_multilabel'")
        self._docs: Optional[List[Doc]] = None
        self._vocab: Optional[Dict[str, Any]] = None

    # ---- vocabulary --------------------------------------------------------
    def vocab(self) -> Dict[str, Any]:
        if self._vocab is None:
            rng = np.random.default_rng(self.vocab_seed * 7919 + 13)
            V = self.vocab_size
            words = []
            seen = set()
            for i in range(V):
                w = _make_word(i, rng)
                while w in seen:
                    w = w + _SYL[int(rng.integers(0, len(_SYL)))]
                seen.add(w)
                words.append(w)
            # a slice of the vocabulary is numeric / punctuation to exercise SHAPE
            for i in range(0, V, 37):
                words[i] = str(int(rng.integers(1, 99999)))
            for i, p in zip(range(5, V, 101), itertools_cycle([".", ",", ";", "!", "?", "-", "(", ")"])):
                words[i] = p
            tag_of = rng.integers(0, self.n_tags, size=V)
            # entity sub-vocabularies: capitalised names, 400 per label
            ent_words: List[List[str]] = []
            for lab in range(self.n_ent_labels):
                names = []
                for k in range(400):
                    base = _make_word(k, rng)
                    names.append(base.capitalize() + ("" if k % 3 else _SYL[lab % len(_SYL)]))
                ent_words.append(names)
            all_words = list(words)
            ent_offset = []
            for names in ent_words:
                ent_offset.append(len(all_words))
                all_words.extend(names)
            attrs = featurize_words(all_words)
            ranks = np.arange(1, V + 1, dtype=np.float64)
            probs = 1.0 / ranks
            probs /= probs.sum()
            self._vocab = {"words": all_words, "attrs": attrs, "tag_of": tag_of, "probs": probs,
                           "ent_offset": ent_offset, "n_base": V}
        return self._vocab

    # ---- documents ---------------------------------------------------------
    def docs(self) -> List[Doc]:
        if self._docs is not None:
            return self._docs
        voc = self.vocab()
        rng = np.random.default_rng(self.seed)
        V = voc["n_base"]
        words_all, attrs_all, tag_of = voc["words"], voc["attrs"], voc["tag_of"]
        propn = TAGS.index("PROPN") if "PROPN" in TAGS[: self.n_tags] else 0
        docs: List[Doc] = []
        lens = rng.integers(self.min_len, self.max_len + 1, size=self.n_docs)
        for n in lens:
            n = int(n)
            ids = rng.choice(V, size=n, p=voc["probs"])
            tags = tag_of[ids].copy()
            ents: List[Tuple[int, int, str]] = []
            if "ner" in self.tasks and self.n_ent_labels > 0:
                t = 0
                while t < n:
                    if rng.random() < self.ent_rate:
                        lab = int(rng.integers(0, self.n_ent_labels))
                        span = int(min(n - t, rng.integers(1, 4)))
                        for k in range(span):
                            ids[t + k] = voc["ent_offset"][lab] + int(rng.integers(0, 400))
                            tags[t + k] = propn
                        ents.append((t, t + span, ENT_LABELS[lab]))
                        t += span + 1
                    else:
                        t += 1
            if self.noise > 0:
                flip = rng.random(n) < self.noise
                tags = np.where(flip, rng.integers(0, self.n_tags, size=n), tags)
            heads = deps = None
            if "parser" in self.tasks:
                root = int(rng.integers(0, n))
                jump = rng.random(n) < 0.3
                heads = []
                for t in range(n):
                    if t == root:
                        heads.append(t)
                    elif t < root:
                        heads.append(root if jump[t] else t + 1)
                    else:
                        heads.append(root if jump[t] else t - 1)
                deps = [
                    "ROOT" if h == t else DEP_LABELS[(int(tags[t]) * 2 + (1 if h > t else 0)) % self.n_dep_labels]
                    for t, h in enumerate(heads)
                ]
            doc = Doc(
                [words_all[i] for i in ids],
                tags=[TAGS[int(t)] for t in tags] if "tagger" in self.tasks else None,
                ents=ents if "ner" in self.tasks else None,
                heads=heads, deps=deps,
                attrs=np.ascontiguousarray(attrs_all[ids]),
            )
            if "textcat" in self.tasks or "textcat_multilabel" in self.tasks:
                doc.cats = doc_cats(ids, "textcat_multilabel" in self.tasks)
            docs.append(doc)
        self._docs = docs
        return docs

    def __call__(self, nlp=None) -> Iterator[Example]:
        for doc in self.docs():
            yield Example.from_doc(doc)

    def __len__(self) -> int:
        return self.n_docs


def itertools_cycle(seq):
    import itertools

    return itertools.cycle(seq)


@registry.readers("spacy_ray_b200.SyntheticCorpus.v1")
def create_synthetic_corpus(n_docs: int = 2000, seed: int = 0, min_len: int = 8, max_len: int = 40,
                            vocab_size: int = 20000, n_tags: int = 17, n_ent_labels: int = 4,
                            n_dep_labels: int = 8, ent_rate: float = 0.12, noise: float = 0.02,
                            tasks: Sequence[str] = ("tagger", "ner", "parser"), vocab_seed: int = 0) -> SyntheticCorpus:
    return SyntheticCorpus(n_docs, seed, min_len, max_len, vocab_size, n_tags, n_ent_labels, n_dep_labels,
                           ent_rate, noise, tasks, vocab_seed)
