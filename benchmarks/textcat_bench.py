"""Textcat in the device-resident engine: docs/s of the flagship NER step, of NER + textcat (one shared
tok2vec, width 256, depth 8), and of textcat alone (CNN / BOW / Ensemble), each on the engine (CUDA-graph
replay of the whole step) and on the generic path (``nlp.update``: the same kernels launched one by one).

Timing: warm-up steps first (every graph bucket captured), then ``--steps`` timed steps.  Each step is
bracketed by CUDA events; a 256 MB buffer is overwritten between steps (outside the events) so no step finds
the previous one's weights / activations in the 126 MB L2.  Batches are token-balanced (every step has the same
row count).  The card name and power limit are read in the same run.  A separate ``torch.profiler`` pass over
a few NER + textcat engine steps gives the textcat kernels' device time per step.

    python benchmarks/textcat_bench.py [--docs 1024] [--steps 50] [--generic-steps 10] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

TOK2VEC = """
@architectures = "spacy.Tok2Vec.v2"

[{path}.embed]
@architectures = "spacy.MultiHashEmbed.v2"
width = 256
attrs = ["NORM","PREFIX","SUFFIX","SHAPE"]
rows = [5000,1000,2500,2500]
include_static_vectors = false

[{path}.encode]
@architectures = "spacy.MaxoutWindowEncoder.v2"
width = 256
depth = 8
window_size = 1
maxout_pieces = 3
"""

BOW = """
@architectures = "spacy.TextCatBOW.v2"
exclusive_classes = true
ngram_size = {ngram}
no_output_layer = false
"""


def textcat_alone(arch: str) -> str:
    """textcat with its own flagship tok2vec (CNN: TextCatReduce mean + max; Ensemble: + BOW n-grams 1-2),
    or the bag of words alone (n-grams 1-2)."""
    head = "[components.textcat.model]\n"
    if arch == "bow":
        model = head + BOW.format(ngram=2)
    elif arch == "cnn":
        model = (head + '@architectures = "spacy.TextCatReduce.v1"\nexclusive_classes = true\nuse_reduce_mean = true\n'
                 'use_reduce_max = true\nuse_reduce_first = false\nuse_reduce_last = false\n\n'
                 "[components.textcat.model.tok2vec]" + TOK2VEC.format(path="components.textcat.model.tok2vec"))
    else:
        model = (head + '@architectures = "spacy.TextCatEnsemble.v2"\nnO = null\n\n'
                 "[components.textcat.model.tok2vec]" + TOK2VEC.format(path="components.textcat.model.tok2vec")
                 + "\n[components.textcat.model.linear_model]" + BOW.format(ngram=2))
    return f"""
[nlp]
lang = "en"
pipeline = ["textcat"]

[components]

[components.textcat]
factory = "textcat"

{model}
[corpora]

[corpora.train]
@readers = "spacy_ray_b200.SyntheticCorpus.v1"
n_docs = 8192
seed = 1
min_len = 8
max_len = 40
tasks = ["textcat"]

[training]
dropout = 0.1
"""


def card() -> dict:
    import torch

    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return out


def _setup(text: str, docs: int):
    from spacy_ray_b200.config import Config
    from spacy_ray_b200.worker import Worker

    cfg = Config().from_str(text, interpolate=False)
    cfg["corpora"]["train"]["n_docs"] = docs * 8
    cfg["training"]["max_steps"] = 0
    w = Worker(cfg, rank=0, num_workers=1, use_gpu=0, mode="sync", comm="auto", fused_ops=True)
    w.set_proxy(None)
    tr = cfg["corpora"]["train"]
    return w, list(w.train_corpus(w.nlp)), docs * (int(tr["min_len"]) + int(tr["max_len"])) // 2


def measure(text: str, docs: int, steps: int, warmup: int, engine: bool, profile_steps: int = 0) -> dict:
    import torch

    from spacy_ray_b200.engine import Trainer

    w, examples, tokens = _setup(text, docs)
    nlp, proxy = w.nlp, w.proxy
    trainer = Trainer(nlp, proxy, examples, docs_per_batch=docs, dropout=0.1, prefetch=False, bucket_rows=128)
    batches = trainer.batches(warmup + steps + profile_steps, seed=0, tokens_per_batch=tokens)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device="cuda")     # 256 MB > L2
    if engine:
        staged = []
        for ids in batches:
            trainer.prepare(ids)
            st = trainer._take()
            staged.append((st["buf"].to(trainer.device), st["rows"]))

        def step(i):
            buf, rows = staged[i]
            trainer.dev_buf.copy_(buf, non_blocking=True)
            return trainer._run(rows)

        step(0)                                                 # eager first step, then capture
        trainer.capture_buckets([r for _b, r in staged])
    else:
        egs = [[examples[i] for i in ids] for ids in batches]

        def step(i):
            losses = {}
            nlp.update(egs[i], drop=0.1, sgd=False, losses=losses)
            proxy.step()
            return losses

    for i in range(1 if engine else 0, warmup):
        step(i)
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.zero_()
        evs[k][0].record()
        step(warmup + k)
        evs[k][1].record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in evs)
    total = sum(ms)
    out = {"docs_per_s": docs * steps / (total / 1e3), "ms_per_step": {"mean": total / steps, "min": ms[0],
                                                                        "median": ms[len(ms) // 2], "max": ms[-1]},
           "engine": engine, "graphs": len(trainer._graphs) if engine else 0, "heads": trainer.loss_names}
    if profile_steps and engine:
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(profile_steps):
                step(warmup + steps + k)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if "textcat" in e.key:
                per[e.key] = {"us_per_step": e.device_time_total / profile_steps, "calls": e.count}
        out["textcat_kernels"] = per
        out["textcat_us_per_step"] = sum(v["us_per_step"] for v in per.values())
    trainer.close()
    w.proxy = None
    del trainer, w, nlp, proxy
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    return out


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=1024, help="docs per step")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--generic-steps", type=int, default=10)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "textcat_bench.py needs a CUDA device"}))
        return 1
    cfgs = ROOT / "configs"
    ner = (cfgs / "ner_w256.cfg").read_text()
    ner_tc = (cfgs / "ner_textcat_w256.cfg").read_text()
    res = {"card": card(), "docs_per_step": args.docs, "steps": args.steps, "warmup": args.warmup,
           "timing": "CUDA events per step, 256 MB overwritten between steps (outside the events), "
                     "token-balanced batches (docs * (min_len + max_len) / 2 tokens)",
           "arms": {}}
    arms = res["arms"]
    arms["ner/engine"] = measure(ner, args.docs, args.steps, args.warmup, True)
    arms["ner+textcat/engine"] = measure(ner_tc, args.docs, args.steps, args.warmup, True,
                                         profile_steps=args.profile_steps)
    arms["ner+textcat/generic"] = measure(ner_tc, args.docs, args.generic_steps, 3, False)
    for arch in ("cnn", "bow", "ensemble"):
        text = textcat_alone(arch)
        arms[f"textcat_{arch}/engine"] = measure(text, args.docs, args.steps, args.warmup, True,
                                                 profile_steps=args.profile_steps)
        arms[f"textcat_{arch}/generic"] = measure(text, args.docs, args.generic_steps, 3, False)
    res["ner+textcat_vs_ner_step"] = (arms["ner+textcat/engine"]["ms_per_step"]["mean"]
                                      / arms["ner/engine"]["ms_per_step"]["mean"])
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
