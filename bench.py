#!/usr/bin/env python
"""Headline benchmark: docs/sec training en tok2vec(HashEmbed+Maxout width 256, depth 8)+NER.

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` (N>1 under torchrun)
prints ONE JSON line from rank 0.  ``value`` = whole-job docs/s, device-timed with CUDA
events over exactly K steps, max over ranks.  ``e2e`` = the same metric through the public
API (``nlp.update`` + ``proxy.step``) including, every step, the pinned-host -> device copy
of that step's inputs and the device -> host read of the loss.

``--impl reference`` runs the UNMODIFIED reference from ``baseline/_ref`` through its own public
API (``spacy_ray.train_cli.ray_train``, ``/root/reference/spacy_ray/train_cli.py:56-91``) - if it
can be imported.  Its dependencies (spaCy, thinc, Ray<1.0) are not installable offline (DESIGN.md
section 0), so the arm tries the import, and when that fails prints the real exception in the
``unavailable`` line and exits 0.  Two *in-repo* comparison arms exist and are labelled as ours:
``--impl nccl-baseline`` (NCCL reduce-scatter/all-gather + cuBLAS GEMMs + unfused per-key torch
Adam + per-op launches) - also run automatically after the product arm at the same N / steps and
reported as ``vs_own_nccl_baseline`` - and ``--impl rayproxy-emu`` (per-key host-staged async
proxy protocol, ``benchmarks/bench_rayproxy.py``).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BASELINE_PUBLISHED = None   # BASELINE.md: the reference publishes no numbers


def flagship_config(args, rank: int) -> str:
    n_docs = args.docs_per_gpu * 8
    return f"""
[system]
seed = 0

[nlp]
lang = "en"
pipeline = ["ner"]

[components]

[components.ner]
factory = "ner"

[components.ner.model]
@architectures = "spacy.TransitionBasedParser.v2"
state_type = "ner"
extra_state_tokens = false
hidden_width = 64
maxout_pieces = 2
use_upper = true

[components.ner.model.tok2vec]
@architectures = "spacy.Tok2Vec.v2"

[components.ner.model.tok2vec.embed]
@architectures = "spacy.MultiHashEmbed.v2"
width = {args.width}
attrs = ["NORM","PREFIX","SUFFIX","SHAPE"]
rows = [5000,1000,2500,2500]
include_static_vectors = false

[components.ner.model.tok2vec.encode]
@architectures = "spacy.MaxoutWindowEncoder.v2"
width = {args.width}
depth = {args.depth}
window_size = 1
maxout_pieces = 3

[corpora]

[corpora.train]
@readers = "spacy_ray_b200.SyntheticCorpus.v1"
n_docs = {n_docs}
seed = {1000 + rank}
min_len = {args.min_len}
max_len = {args.max_len}
n_ent_labels = 18
tasks = ["ner"]

[corpora.dev]
@readers = "spacy_ray_b200.SyntheticCorpus.v1"
n_docs = 64
seed = 7
min_len = {args.min_len}
max_len = {args.max_len}
n_ent_labels = 18
tasks = ["ner"]

[training]
dropout = {args.dropout}
max_steps = 0
"""


def reference_arm(args) -> int:
    """Run the unmodified reference (baseline/_ref) on its own code path, or say exactly why not."""
    ref_dir = ROOT / "baseline" / "_ref"
    line = {"impl": "reference", "n_gpus": args.gpus}
    if not (ref_dir / "spacy_ray").is_dir():
        line["unavailable"] = (f"{ref_dir}/spacy_ray does not exist (pip install --no-index --no-deps --target "
                               "baseline/_ref /root/reference has not been run on this box)")
        print(json.dumps(line))
        return 0
    sys.path.insert(0, str(ref_dir))
    try:
        import importlib

        mod = importlib.import_module("spacy_ray")              # noqa: F841  (imports spacy, thinc, typer)
        from spacy_ray.train_cli import ray_train                # noqa: F401
        import ray                                                # noqa: F401
    except BaseException as e:                                    # ImportError, or whatever the import chain raises
        missing = []
        for dep in ("spacy", "thinc", "ray", "typer", "wasabi", "srsly"):
            try:
                importlib.import_module(dep)
            except BaseException:
                missing.append(dep)
        line["unavailable"] = (f"import spacy_ray from {ref_dir} failed: {type(e).__name__}: {e}; "
                               f"not importable here: {', '.join(missing) or 'none'} "
                               "(no wheels in /opt/wheelhouse, no network; ray<1.0 has no cp312 build)")
        print(json.dumps(line))
        return 0
    # The reference imported: drive its stock path (ray_train -> Ray Worker actors -> spaCy's
    # train_while_improving) on the flagship config.  It exposes no step hook and discards the model,
    # so docs/s comes from the wall-clock difference of two runs (W and W + K steps) - its start-up
    # (ray.init, actor creation, init_nlp on every worker) cancels out.
    try:
        line.update(_drive_reference(args, ray_train))
    except BaseException as e:
        line["unavailable"] = f"reference imported but could not be driven: {type(e).__name__}: {e}"
    print(json.dumps(line))
    return 0


REFERENCE_CFG = """
[paths]
train = "{train}"
dev = "{dev}"

[nlp]
lang = "en"
pipeline = ["ner"]

[components]

[components.ner]
factory = "ner"

[components.ner.model]
@architectures = "spacy.TransitionBasedParser.v2"
state_type = "ner"
extra_state_tokens = false
hidden_width = 64
maxout_pieces = 2
use_upper = true

[components.ner.model.tok2vec]
@architectures = "spacy.Tok2Vec.v2"

[components.ner.model.tok2vec.embed]
@architectures = "spacy.MultiHashEmbed.v2"
width = {width}
attrs = ["NORM","PREFIX","SUFFIX","SHAPE"]
rows = [5000,1000,2500,2500]
include_static_vectors = false

[components.ner.model.tok2vec.encode]
@architectures = "spacy.MaxoutWindowEncoder.v2"
width = {width}
depth = {depth}
window_size = 1
maxout_pieces = 3

[corpora.train]
@readers = "spacy.Corpus.v1"
path = ${{paths.train}}

[corpora.dev]
@readers = "spacy.Corpus.v1"
path = ${{paths.dev}}

[training]
dropout = {dropout}
max_steps = {max_steps}
eval_frequency = 1000000
patience = 0

[training.batcher]
@batchers = "spacy.batch_by_sequence.v1"
size = {batch}
get_length = null
"""


def _drive_reference(args, ray_train) -> dict:
    import tempfile
    import time

    from spacy import util as spacy_util                         # the reference's own config loader
    from spacy_ray_b200.training.corpus import SyntheticCorpus
    from spacy_ray_b200.training.docbin import DocBin

    tmp = Path(tempfile.mkdtemp(prefix="srb_ref_"))
    n_docs = args.docs_per_gpu * 8
    for name, n, seed in (("train", n_docs, 1000), ("dev", 64, 7)):
        corpus = SyntheticCorpus(n, seed=seed, min_len=args.min_len, max_len=args.max_len, n_ent_labels=18, tasks=("ner",))
        DocBin(docs=corpus.docs()).to_disk(tmp / f"{name}.spacy")

    def run(steps: int) -> float:
        text = REFERENCE_CFG.format(train=tmp / "train.spacy", dev=tmp / "dev.spacy", width=args.width, depth=args.depth,
                                    dropout=args.dropout, max_steps=steps, batch=args.docs_per_gpu)
        cfg_path = tmp / f"ref_{steps}.cfg"
        cfg_path.write_text(text)
        config = spacy_util.load_config(cfg_path, interpolate=False)
        t0 = time.perf_counter()
        ray_train(config, num_workers=args.gpus, use_gpu=0)
        return time.perf_counter() - t0

    w, k = max(args.warmup, 3), args.steps
    t_w = run(w)
    t_wk = run(w + k)
    dt = max(t_wk - t_w, 1e-9)
    docs = float(k * args.docs_per_gpu * args.gpus)       # every worker consumes a batch per step
    return {"metric": "docs/sec (whole box) en tok2vec+NER", "value": docs / dt, "unit": "docs/s", "steps": k, "warmup": w,
            "ms_per_step": dt / k * 1e3, "timing": "wall clock, difference of a (W+K)-step and a W-step run",
            "dtype": "fp32 (thinc default)", "data": "synthetic (same generator, written as DocBin)"}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, losses, proxy) -> None:
    """Write what the last timed step hands its caller: ``losses.npy`` (per-head losses, ``loss_names`` order)
    and ``params.npy`` (every parameter after the optimizer update, layout order, padding left out), both
    float32.  Parameters beyond the byte budget are replaced by a fixed, seeded sample of them.  The inputs are
    seeded, but some device sums accumulate in a varying order: two runs agree to rounding after a few steps and
    drift apart over hundreds, so compare two builds at a small ``--steps``."""
    import numpy as np
    import torch

    lay = proxy.layout
    idx = torch.cat([torch.arange(lay.offset[k], lay.offset[k] + lay.numel[k]) for k in lay.keys])
    cap = (DUMP_BYTES - 4 * losses.numel()) // 4
    if idx.numel() > cap:
        pick = np.sort(np.random.default_rng(0).choice(idx.numel(), size=cap, replace=False))
        idx = idx[torch.from_numpy(pick)]
    params = proxy.param_flat[idx.to(proxy.param_flat.device)].float().cpu().numpy()
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "losses.npy", losses.detach().float().cpu().numpy())
    np.save(out / "params.npy", params)


def run_arm(args, impl: str, rank: int, world: int, local_rank: int, steps: int, dump_dir=None):
    """One measured arm (``ours`` / ``nccl-baseline``) of ``steps`` timed steps.  Returns the result dict on
    every rank.  With ``dump_dir``, rank 0 writes the outputs of the last timed step there (``dump_outputs``)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from spacy_ray_b200.config import Config
    from spacy_ray_b200.utils.timing import ClockSampler
    from spacy_ray_b200.worker import Worker

    if impl == "nccl-baseline":
        os.environ["SRB_USE_TC"] = "0"          # cuBLAS GEMMs, library collectives, per-key torch Adam
    else:
        os.environ.pop("SRB_USE_TC", None)
    comm = args.comm
    if impl == "nccl-baseline":
        comm = "local" if world == 1 else "dist"
    min_len, max_len = args.min_len, args.max_len
    if args.config:
        cfg = Config().from_str(Path(args.config).read_text(), interpolate=False)
        cfg["corpora"]["train"]["n_docs"] = args.docs_per_gpu * 8
        cfg["corpora"]["train"]["seed"] = 1000 + rank
        cfg["training"]["max_steps"] = 0
        min_len = int(cfg["corpora"]["train"].get("min_len", min_len))
        max_len = int(cfg["corpora"]["train"].get("max_len", max_len))
    else:
        cfg = Config().from_str(flagship_config(args, rank), interpolate=False)
    worker = Worker(cfg, rank=rank, num_workers=world, use_gpu=local_rank, mode="sync", comm=comm,
                    fused_ops=True)
    worker.set_proxy(None)
    nlp, proxy = worker.nlp, worker.proxy
    from spacy_ray_b200.ops import get_current_ops

    ops = get_current_ops()
    examples = list(worker.train_corpus(nlp))
    B = args.docs_per_gpu
    n_params = sum(proxy.layout.numel.values())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    from spacy_ray_b200.engine import Trainer

    use_graphs = args.engine == "graph" and impl == "ours"
    trainer = Trainer(nlp, proxy, examples, docs_per_batch=B, dropout=args.dropout, use_graphs=use_graphs,
                      bucket_rows=args.bucket_rows)
    warmup = args.warmup
    n_total = warmup + steps
    # token-balanced batches: every rank's every batch holds exactly B * (min_len + max_len) / 2 tokens,
    # so all ranks run the same row count each step (a synchronous step is as slow as its largest batch)
    tokens = None if args.random_batches else B * (min_len + max_len) // 2
    id_batches = trainer.batches(2 * n_total + 2, seed=rank, tokens_per_batch=tokens)

    # ---------------- device-timed: inputs already on the device, no host reads ----------------
    # (each step's packed input block is staged on the device beforehand and moved into the
    #  static input buffer with a D2D copy inside the timed region)
    dev_inputs = []
    for ids in id_batches[:n_total]:
        trainer.prepare(ids)
        stage = trainer._take()
        dev_inputs.append((stage["buf"].to(trainer.device), stage["rows"], stage["docs"], stage["words"]))
    torch.cuda.synchronize()

    def device_step(item):
        packed, rows, _d, _w = item
        trainer.dev_buf.copy_(packed, non_blocking=True)
        return trainer._run(rows)

    device_step(dev_inputs[0])                       # first step runs eagerly on every rank
    trainer.capture_buckets([it[1] for it in dev_inputs] +
                            [trainer.rows_for(ids) for ids in id_batches[n_total:]])
    for item in dev_inputs[1: warmup]:
        device_step(item)
    launches0 = ops.launches + getattr(proxy.comm, "launches", 0)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    # the sampler thread (NVML init, ~ms, different on every rank) starts BEFORE the barrier: the start
    # event must follow the barrier immediately, or the rank that gets going first spends the difference
    # waiting for its peers inside its first timed step and max-over-ranks reports start skew as step time
    with ClockSampler(local_rank) as clocks:
        barrier()
        evs[0].record()
        for i, item in enumerate(dev_inputs[warmup: n_total]):
            losses = device_step(item)
            evs[i + 1].record()
        barrier()
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, losses, proxy)
    ms = max_over_ranks(float(evs[0].elapsed_time(evs[-1])))
    per_step = sorted(float(evs[i].elapsed_time(evs[i + 1])) for i in range(steps))
    launches = ops.launches + getattr(proxy.comm, "launches", 0) - launches0
    docs = sum_over_ranks(float(sum(it[2] for it in dev_inputs[warmup: n_total])))
    words = sum_over_ranks(float(sum(it[3] for it in dev_inputs[warmup: n_total])))
    value = docs / (ms / 1e3)
    if hasattr(proxy.comm, "check"):
        proxy.comm.check()

    # ---------------- end to end through the public API -----------------------------------------
    # Trainer.train_step(): native collate into pinned memory (prefetch thread) -> ONE H2D copy
    # -> CUDA-graph replay of the whole step -> D2H copy of the per-head losses.  Every step; the host
    # reads each loss one step late (it is logging data) so the device never waits for the host.
    e2e = None
    if args.e2e:
        rest = id_batches[n_total: 2 * n_total + 2]
        state = {"next": 0, "ahead": 0}

        def top_up():
            # the batch about to run + `trainer.prefetch_depth` more being collated behind it (the trainer
            # raises the depth from 1 to its number of collate workers when the device waited for the host)
            while state["ahead"] < trainer.prefetch_depth + 1 and state["next"] < len(rest):
                trainer.prepare(rest[state["next"]])
                state["next"] += 1
                state["ahead"] += 1

        for i in range(warmup):
            top_up()
            trainer.train_step()
            state["ahead"] -= 1
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        docs_local = 0
        with ClockSampler(local_rank) as clocks_e:
            barrier()
            e0.record()
            for i in range(warmup, n_total):
                top_up()                              # collate FUTURE batches while this one runs
                loss_val = trainer.train_step()       # H2D + step + async D2H(loss); returns the previous step's
                state["ahead"] -= 1
                docs_local += trainer.last["docs"]
            loss_val = trainer.flush_loss()           # the last step's loss is read inside the timed region too
            e1.record()
            barrier()
        ms_e = max_over_ranks(float(e0.elapsed_time(e1)))
        docs_e = sum_over_ranks(float(docs_local))
        e2e = {"value": docs_e / (ms_e / 1e3), "unit": "docs/s", "h2d_bytes_per_step": int(trainer.h2d_bytes_per_step),
               "d2h_bytes_per_step": 4 * len(trainer.loss_names), "ms_per_step": ms_e / steps, "last_loss": loss_val,
               "api": "spacy_ray_b200.engine.Trainer.train_step",
               "timed_region": "per step: native collate of the batch from the pre-featurised in-memory ExampleStore "
                               "(prefetch thread) -> pinned buffer -> H2D -> graph replay -> D2H of the losses; "
                               "tokenisation / attribute hashing of the corpus happen once, before the timed region",
               "clocks": clocks_e.summary()}
        if hasattr(proxy.comm, "check"):
            proxy.comm.check()
    trainer.close()
    mean_len = words / max(docs, 1)
    out = {
        "metric": "docs/sec (whole box, device-timed, max over ranks) "
                  + ("en tok2vec+NER" if not args.config else "+".join(nlp.pipe_names)),
        "value": value, "unit": "docs/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic (SyntheticCorpus, random-init weights)",
        "impl": impl, "engine": args.engine if impl == "ours" else "eager",
        "config": {
            "model": (f"en tok2vec(MultiHashEmbed+MaxoutWindowEncoder width={args.width} depth={args.depth})+NER "
                      f"(TransitionBasedParser hidden=64, 18 entity labels)") if not args.config
            else f"{args.config} pipeline={nlp.pipe_names}",
            "global_batch": int(B * world), "docs_per_gpu": B, "seq_len": round(mean_len, 2),
            "words_per_sec": words / (ms / 1e3), "params": int(n_params),
            "parallelism": f"dp{world} + optimizer sharding by parameter ownership ({proxy.comm.name})",
            "batching": ("random docs per batch" if tokens is None else
                         f"token-balanced: every batch = {B} docs / {tokens} tokens on every rank"),
            "l2": "per-step inputs + activations exceed the 126 MB L2 (fresh batch every step)",
            "optimizer": "Adam (thinc semantics, per-tensor clip 1.0, wd 0.01), fp32 master",
            "exchange_buckets": getattr(getattr(proxy.comm, "plan", None), "n", None),
            "shard_balance": worker._balance(),
        },
        "step_ms": {"min": per_step[0], "median": per_step[len(per_step) // 2], "max": per_step[-1]},
        "clocks": clocks.summary(),
        "e2e": e2e,
        "gpu_launches": int(launches),
    }
    # free the symmetric buffers / graphs before a second arm is built in this process
    worker.proxy = None
    del trainer, worker, proxy, nlp
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    return out


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl-baseline", "rayproxy-emu"])
    ap.add_argument("--docs-per-gpu", type=int, default=1024)
    ap.add_argument("--width", type=int, default=256)
    ap.add_argument("--depth", type=int, default=8)
    ap.add_argument("--min-len", type=int, default=8)
    ap.add_argument("--max-len", type=int, default=40)
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--no-e2e", dest="e2e", action="store_false")
    ap.add_argument("--comm", default="auto")
    ap.add_argument("--config", default=None,
                    help="train a pipeline from a .cfg file (configs/*.cfg) instead of the flagship tok2vec+NER; "
                         "its [corpora.train] must be a SyntheticCorpus (n_docs/seed are overridden per rank)")
    ap.add_argument("--engine", default="graph", choices=["graph", "eager"],
                    help="graph = CUDA-graph replay of the whole step; eager = same kernels launched from Python")
    ap.add_argument("--bucket-rows", type=int, default=128, help="row granularity of the captured graphs")
    ap.add_argument("--random-batches", action="store_true",
                    help="plain random batches (row counts differ between ranks and steps) instead of token-balanced ones")
    ap.add_argument("--no-own-baseline", dest="own_baseline", action="store_false",
                    help="skip the nccl-baseline arm that is otherwise run after the product arm")
    ap.add_argument("--baseline-steps", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the losses and updated parameters of the last one to "
                         "DIR/*.npy (float32, at most 64 MB) so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        return reference_arm(args)

    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "bench.py needs a CUDA device", "impl": args.impl}))
        return 1
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    import torch.distributed as dist

    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    if args.impl == "rayproxy-emu":
        print(json.dumps({"impl": args.impl, "unavailable": "rayproxy-emu runs under the actor runtime: "
                          "use benchmarks/bench_rayproxy.py"}))
        return 0
    out = run_arm(args, args.impl, rank, world, local_rank, args.steps, dump_dir=args.dump_outputs)
    if args.impl == "ours" and args.own_baseline:
        # OUR emulation of an NCCL(+cuBLAS) build of the reference's data flow, same box, same N, same
        # metric/config - context for the reader; the published-number ratio `vs_baseline` stays null
        # because the reference publishes nothing (BASELINE.md)
        try:
            base = run_arm(args, "nccl-baseline", rank, world, local_rank, min(args.steps, args.baseline_steps))
            out["vs_own_nccl_baseline"] = {
                "ratio": out["value"] / base["value"], "baseline_value": base["value"], "baseline_steps": base["steps"],
                "baseline_ms_per_step": base["ms_per_step"],
                "what": "this repo's --impl nccl-baseline arm (NCCL reduce-scatter/all-gather, cuBLAS GEMMs, per-key "
                        "torch Adam, per-op launches) - our emulation, NOT the reference's number",
            }
        except Exception as e:                   # never lose the product line to the context arm
            out["vs_own_nccl_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
