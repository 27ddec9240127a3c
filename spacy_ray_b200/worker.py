"""``Worker``: one training process per rank (and ``Evaluator``, ``FakeOptimizer``,
``thread_training``).

Same public surface as ``/root/reference/spacy_ray/worker.py`` - constructor
``Worker(config, *, rank, num_workers, use_gpu, code_path, ray)``; control plane
``set_proxy / train / is_running / evaluate / save_checkpoint / get_owned_keys /
get_peer_map / sync_params / get_percent_grads_used / get_quorum``; data plane
``inc_grad / set_param / get_param`` - but usable three ways:

1. as an actor under the built-in runtime (``parallel/actors.py``), driven by
   ``ray_train`` exactly like the reference drives Ray actors;
2. SPMD under ``torchrun`` (one ``Worker`` per process, ``peers=None``), which is
   how ``bench.py`` runs;
3. in-process, several workers wired together directly (unit tests).

Communication ``mode``:

``"async"``  the reference protocol (``PeerProxy``): per-key versioned pushes,
             quorum default 2 (``proxies.py:33``), host-staged messages.
``"sync"``   flat-bucket reduce-scatter -> sharded Adam -> all-gather once per
             step (``ShardedSyncProxy``), over ``torch.distributed`` ("dist":
             NCCL/gloo - the baseline) or the fused sm_100a peer-memory kernel
             ("fused" - the product).  Quorum = num_workers x accumulate_gradient,
             the value ``get_quorum`` (``worker.py:151-155``) computes.

Fixes relative to the reference (SURVEY.md 0.7-0.8): checkpoints are written
(``--output``), per-rank data sharding, training-thread exceptions surface,
score sharing is step-indexed, grads-used counters are real.
"""
from __future__ import annotations

import os
import threading
import time
import traceback
from pathlib import Path
from typing import Any, Callable, Dict, List, Optional, Union

import torch

from .config import Config, registry, resolve_dot_names
from .nn.layers import offset_dropout_stream
from .ops import get_current_ops, require_cpu, require_gpu, set_current_ops
from .parallel.proxies import PeerProxy, RayPeerProxy  # noqa: F401
from .parallel.sync_proxy import FlatLayout, LocalComm, ShardedSyncProxy, TorchDistComm
from .parallel.util import DIVIDERS, KeyT, set_params_proxy
from .training.checkpoint import load_optimizer_shards, save_optimizer_shard, save_pipeline
from .training.initialize import init_nlp
from .training.loop import (
    ConfigSchemaTraining, create_before_to_disk_callback, create_evaluation_callback,
    create_train_batches, train_while_improving,
)
from .utils.logging import logger
from .utils.code import import_code


class Worker:
    rank: int
    num_workers: int
    gpu_id: int

    def __init__(
        self,
        config: Union[Config, Dict[str, Any]],
        *,
        rank: int = 0,
        num_workers: int = 1,
        use_gpu: int = 0,
        code_path: Optional[Path] = None,
        ray: Any = None,
        mode: str = "sync",
        comm: str = "auto",
        quorum: Optional[int] = None,
        output_path: Optional[Path] = None,
        resume_path: Optional[Path] = None,
        shard_data: bool = True,
        shard_balance: str = "auto",
        grad_transport: str = "fp32",
        dist_init: Optional[Dict[str, Any]] = None,
        fused_ops: bool = True,
        inject_fault: Optional[str] = None,
    ):
        if ray is None:
            from .parallel import actors as ray  # built-in runtime with Ray's surface
        self.ray = ray
        import_code(code_path)
        self.rank = rank
        self.num_workers = num_workers
        self.mode = mode
        self.comm_name = comm
        self.quorum = quorum
        self.output_path = Path(output_path) if output_path else None
        self.resume_path = Path(resume_path) if resume_path else None
        self.shard_data = shard_data
        self.shard_balance = shard_balance
        self.grad_transport = grad_transport
        self.dist_init = dict(dist_init or {})
        self.inject_fault = inject_fault
        self.gpu_id = self._resolve_gpu(use_gpu, fused_ops)
        self.nlp = init_nlp(Config(config), use_gpu=-1)   # ops already selected above
        config = self.nlp.config.interpolate()
        self.config = config
        self.T = registry.resolve(config["training"], schema=ConfigSchemaTraining)
        dot_names = [self.T["train_corpus"], self.T["dev_corpus"]]
        self.train_corpus, self.dev_corpus = resolve_dot_names(config, dot_names)
        self.before_to_disk = create_before_to_disk_callback(self.T["before_to_disk"])
        if num_workers > 1:
            offset_dropout_stream(rank)
        self._evaluation_callback: Callable = lambda: (0.0, {})
        self._has_evaluation_callback = False
        self._results: List = []
        self.thread: Optional[threading.Thread] = None
        self.proxy: Any = None
        self.optimizer = None
        self._error: Optional[str] = None
        self._last_info: Optional[Dict[str, Any]] = None
        self._eval_index = 0
        self._stats: Dict[str, Any] = {"steps": 0, "skip": 3, "docs": 0, "words": 0, "t0": 0.0, "t1": 0.0}
        self._dist_ready = False
        self.n_grads_used = 0
        self.n_grads_discarded = 0

    # ------------------------------------------------------------------ data plane (async mode)
    def inc_grad(self, key: KeyT, version: int, value: torch.Tensor) -> None:
        if self.proxy is None:
            raise ValueError("Proxy object not set")
        key = tuple(key)
        if hasattr(self.proxy, "receive_grad"):
            self.proxy.receive_grad(key, version, value)
        elif self.proxy.check_version(key, version):
            self.proxy.inc_grad(key[0], key[1], value)

    def set_param(self, key: KeyT, version: int, value: torch.Tensor) -> None:
        if self.proxy is None:
            raise ValueError("Proxy object not set")
        return self.proxy.receive_param(tuple(key), version, value)

    def get_param(self, key: KeyT, version: int) -> Optional[torch.Tensor]:
        if self.proxy is None:
            raise ValueError("Proxy object not set")
        key = tuple(key)
        if self.proxy.check_version(key, version):
            return self.proxy.get_param(key[0], key[1])
        return None

    # ------------------------------------------------------------------ control plane
    def sync_params(self) -> None:
        if isinstance(self.proxy, ShardedSyncProxy):
            self.proxy.sync_from_owner()
        else:
            for key in list(self.proxy._owned_keys):
                self.proxy.send_param(key)

    def get_percent_grads_used(self) -> Optional[float]:
        if self.proxy is not None:
            self.n_grads_used = self.proxy.n_grads_used
            self.n_grads_discarded = self.proxy.n_grads_discarded
        total = self.n_grads_used + self.n_grads_discarded
        return None if total == 0 else self.n_grads_used / total

    def get_quorum(self) -> int:
        return self.num_workers * int(self.T["accumulate_gradient"])

    def _balance(self) -> str:
        """``auto``: the reference partition (node counts, leftovers to the last rank) everywhere except
        under the fused exchange, whose step time is set by the heaviest shard -> size-balanced."""
        if self.shard_balance != "auto":
            return self.shard_balance
        return "lpt" if self._resolved_comm() == "fused" else "nodes"

    def _resolved_comm(self) -> str:
        if self.mode != "sync":
            return "actors"
        if self.comm_name != "auto":
            return self.comm_name
        ops = get_current_ops()
        if ops.device.type == "cuda" and getattr(ops, "fused", False):
            return "fused"                    # bucketed RS+Adam+AG kernels (also the 1-GPU multi-tensor optimizer)
        return "local" if self.num_workers == 1 else "dist"

    def _divide(self, model):
        return DIVIDERS[self._balance()](model, self.num_workers)

    def get_owned_keys(self) -> List[KeyT]:
        owned: List[KeyT] = []
        for _name, component in self.nlp.pipeline:
            if hasattr(component, "model"):
                owned.extend(self._divide(component.model)[self.rank])
        return owned

    def get_peer_map(self, workers) -> Dict[KeyT, Any]:
        peer_map: Dict[KeyT, Any] = {}
        for _name, component in self.nlp.pipeline:
            if hasattr(component, "model"):
                for worker, keys in zip(workers, self._divide(component.model)):
                    for key in keys:
                        peer_map[key] = worker
        return peer_map

    def _ensure_dist(self) -> None:
        if self._dist_ready or self.num_workers == 1:
            return
        import torch.distributed as dist

        if not dist.is_initialized():
            info = self.dist_init
            backend = info.get("backend") or ("nccl" if get_current_ops().device.type == "cuda" else "gloo")
            addr = info.get("master_addr", os.environ.get("MASTER_ADDR", "127.0.0.1"))
            port = int(info.get("master_port", os.environ.get("MASTER_PORT", 29511)))
            kwargs: Dict[str, Any] = {}
            if backend == "nccl":
                kwargs["device_id"] = get_current_ops().device
            dist.init_process_group(
                backend, init_method=f"tcp://{addr}:{port}", rank=self.rank, world_size=self.num_workers, **kwargs
            )
        self._dist_ready = True

    def set_proxy(self, peers=None) -> None:
        """Install the parameter proxy on every component model."""
        self.optimizer = self.T["optimizer"]
        ops = get_current_ops()
        if getattr(self.optimizer, "ops", None) is None:
            self.optimizer.ops = ops
        models = [(name, c.model) for name, c in self.nlp.pipeline if hasattr(c, "model")]
        if self.mode == "async":
            if peers is None:
                raise ValueError("mode='async' needs the list of peer worker handles")
            proxy: Any = PeerProxy(
                self.get_peer_map(peers), self.optimizer, self.get_owned_keys(),
                grads_per_update=self.quorum or 2, ray=self.ray,
                stage_to_host=(ops.device.type == "cuda"),
                all_peers=list(peers), self_index=self.rank,
            )
        elif self.mode == "sync":
            comm_name = self._resolved_comm()
            layout = FlatLayout.build(models, self.num_workers, balance=self._balance())
            buffers = None
            if comm_name == "local":
                comm: Any = LocalComm(self.rank, self.num_workers)
            elif comm_name == "dist":
                self._ensure_dist()
                comm = TorchDistComm(self.rank, self.num_workers, grad_transport=self.grad_transport)
            elif comm_name == "fused":
                if self.grad_transport != "fp32":
                    logger.warning("--grad-transport %s applies to --comm dist; the fused peer-memory exchange "
                                   "moves fp32 gradients", self.grad_transport)
                if self.num_workers > 1:
                    self._ensure_dist()
                from .parallel.fused_comm import FusedSymmComm

                comm = FusedSymmComm(self.rank, self.num_workers, layout, ops.device, optimizer=self.optimizer,
                                     ops=ops)
                buffers = comm.buffers
                ops.gate_provider = comm          # consumer-side gates on freshly exchanged weights (C2)
            else:
                raise ValueError(f"Unknown comm backend {comm_name!r}")
            param_dtype = getattr(ops, "param_dtype", ops.dtype)
            proxy = ShardedSyncProxy(
                layout, self.optimizer, rank=self.rank, world_size=self.num_workers, device=ops.device,
                comm=comm, param_dtype=param_dtype, buffers=buffers,
            )
            if hasattr(comm, "bind"):
                comm.bind(proxy)
        else:
            raise ValueError(f"Unknown mode {self.mode!r} (expected 'sync' or 'async')")
        for _name, model in models:
            set_params_proxy(model, proxy)
        self.proxy = proxy
        if isinstance(proxy, ShardedSyncProxy) and self.num_workers > 1:
            proxy.sync_from_owner()      # everyone starts from the owners' weights
        if self.resume_path is not None:
            self._resume()

    def _resume(self) -> None:
        path = self.resume_path
        assert path is not None
        self.nlp.from_disk(path)
        force = getattr(self.proxy, "load_param", None)      # async proxy: overwrite non-owned keys too
        for _n, c in self.nlp.pipeline:          # push loaded weights through the proxy
            if hasattr(c, "model"):
                for node in c.model.walk():
                    for pname in node.param_names:
                        if node.has_param(pname):
                            value = node._params._params[(node.id, pname)]
                            if force is not None:
                                force(node.id, pname, value, version=2)
                            else:
                                self.proxy.set_param(node.id, pname, value)
        try:
            loaded = load_optimizer_shards(path, self.nlp, self.optimizer, self.get_owned_keys(),
                                           rank=self.rank, world_size=self.num_workers)
        except FileNotFoundError:
            logger.warning("resume: no optimizer shards found under %s; starting with fresh moments", path)
            loaded = None
        proxy = self.proxy
        if loaded is not None and isinstance(proxy, ShardedSyncProxy):
            # fp32 master weights of the owned shard (the checkpointed model holds bf16-rounded values)
            for key, value in (loaded.get("master") or {}).items():
                view = proxy._master_views.get(key)
                if view is not None:
                    view.copy_(value.to(device=view.device, dtype=torch.float32).reshape(view.shape))
            proxy.version = int((loaded.get("extra") or {}).get("version") or 0)
            restore = getattr(proxy.comm, "load_optimizer_state", None)
            if restore is not None:
                restore(loaded["nr_update"])           # device-side update counter (bias correction)
        if isinstance(proxy, ShardedSyncProxy) and self.num_workers > 1:
            proxy.sync_from_owner()

    def train(self, peers=None, evaluator: Any = None) -> None:
        """Build the step generator and start it on a thread (so that, as an
        actor, the main thread keeps serving peers' pushes)."""
        self._evaluator = evaluator

        def evaluate():
            self._eval_index += 1
            if self.rank == 0:
                scores = self.evaluate()
                if evaluator is not None:
                    self._call(evaluator.set_scores, scores, self._eval_index)
                return scores
            if evaluator is None:
                return self.evaluate()
            scores = None
            while scores is None:
                scores = self._call(evaluator.get_scores, self._eval_index)
                if scores is None:
                    time.sleep(0.05)
            return scores

        train_batches = create_train_batches(
            self.nlp, self.train_corpus, self.T["batcher"], self.T["max_epochs"],
            rank=self.rank, world_size=self.num_workers, shard=self.shard_data,
            seed=int(self.T.get("seed") or 0),
        )
        after_step = None
        if isinstance(self.proxy, ShardedSyncProxy):
            self._maybe_install_trainer()

            def after_step(step: int) -> None:
                if self.inject_fault and self.inject_fault == f"{self.rank}:{step}":
                    raise RuntimeError(f"injected fault on rank {self.rank} at step {step}")
                if getattr(self.nlp, "_trainer_stepped", False):
                    self.nlp._trainer_stepped = False      # exchange + optimizer ran inside the graph
                else:
                    self.proxy.step()
        self.training_step_iterator = train_while_improving(
            self.nlp,
            FakeOptimizer(self.optimizer),
            train_batches,
            evaluate=evaluate,
            dropout=self.T["dropout"],
            accumulate_gradient=1 if self.mode == "async" else int(self.T["accumulate_gradient"]),
            patience=self.T["patience"],
            max_steps=self.T["max_steps"],
            eval_frequency=self.T["eval_frequency"],
            exclude=self.T["frozen_components"],
            annotating_components=self.T["annotating_components"],
            before_update=self.T["before_update"],
            after_step=after_step,
        )
        if self.rank == 0:
            print_row, self._finalize_logger = self.T["logger"](self.nlp)
        else:
            print_row, self._finalize_logger = (lambda info: None), (lambda: None)
        self.thread = threading.Thread(
            target=self._thread_main,
            args=(self.training_step_iterator, print_row),
            daemon=True,
        )
        self.thread.start()

    def _maybe_install_trainer(self) -> None:
        """On the B200 backend with the fused comm, serve ``nlp.update`` from the
        device-resident engine when the pipeline is one it supports (any mix of tok2vec /
        tagger / ner / parser / textcat components whose heads fit the device kernels).
        ``SRB_FAST_PATH=0`` keeps the generic per-op path."""
        ops = get_current_ops()
        if os.environ.get("SRB_FAST_PATH", "1") == "0" or not getattr(ops, "fused", False):
            return
        if getattr(self.proxy.comm, "name", "") != "fused":
            return
        if set(self.T["frozen_components"]) or set(self.T["annotating_components"]):
            return
        try:
            from .engine import Trainer

            why = Trainer.unsupported_reason(self.nlp)
            if why is not None:
                logger.info("rank %d: generic training path (%s)", self.rank, why)
                return
            # The store is sized from (a sample of) the corpus.  A finite corpus is indexed whole - its
            # batches are then collated by doc id on the native path; a streamed corpus (max_epochs = -1)
            # or one beyond SRB_FAST_PATH_STORE_DOCS contributes only its first docs, and batches of
            # unseen docs go through a throw-away per-batch store (Trainer.update_examples).
            import itertools

            limit = int(os.environ.get("SRB_FAST_PATH_STORE_DOCS", 2_000_000))
            if int(self.T["max_epochs"]) < 0:
                limit = min(limit, int(os.environ.get("SRB_FAST_PATH_SAMPLE", 4096)))
            examples = list(itertools.islice(self.train_corpus(self.nlp), limit))
            if not examples:
                return
            cap = int(os.environ.get("SRB_FAST_PATH_MAX_DOCS", 2048))
            acc = int(self.T["accumulate_gradient"])
            self.nlp._trainer = Trainer(self.nlp, self.proxy, examples, docs_per_batch=min(cap, len(examples)),
                                        dropout=float(self.T["dropout"]), prefetch=False,
                                        exchange=(acc <= 1),      # accumulate_gradient > 1: exchange once per full batch
                                        # (with peers the per-step accumulator clear must not be replayed for
                                        #  every micro-batch: same kernels, launched eagerly)
                                        use_graphs=(acc <= 1 or self.num_workers == 1))
            logger.info("rank %d: device-resident training engine enabled", self.rank)
        except Exception as e:       # never fatal: the generic path is always available
            logger.warning("rank %d: fast path unavailable (%s); using the generic path", self.rank, e)

    def _thread_main(self, iterator, print_row) -> None:
        try:
            thread_training(
                iterator, print_row, self.rank, self.num_workers, self.gpu_id,
                on_step=self._on_step, ops=get_current_ops(),
            )
            if self.output_path is not None and self._last_info is not None:
                self.save_checkpoint(self._last_info, self.output_path / "model-last")
            self._finalize_logger()
        except BaseException:
            self._error = traceback.format_exc()
            logger.error("training thread of rank %d failed:\n%s", self.rank, self._error)

    def _on_step(self, batch, info, is_best_checkpoint) -> None:
        self._last_info = info
        now = time.perf_counter()
        st = self._stats
        if st["steps"] == st["skip"]:               # start the clock after the warm-up steps
            st["t0"], st["docs"], st["words"] = now, 0, 0
        elif st["steps"] > st["skip"]:
            st["docs"] += len(batch)
            st["words"] += sum(len(eg) for eg in batch)
            st["t1"] = now
        st["steps"] += 1
        if is_best_checkpoint and self.output_path is not None:
            self.save_checkpoint(info, self.output_path / "model-best")

    def get_stats(self) -> Dict[str, Any]:
        """Wall-clock throughput of this rank's training thread (steps after the first few)."""
        st = dict(self._stats)
        dt = max(st.get("t1", 0.0) - st.get("t0", 0.0), 1e-9)
        st["seconds"] = dt
        st["docs_per_sec"] = st["docs"] / dt
        st["words_per_sec"] = st["words"] / dt
        proxy = self.proxy
        st["grads_used"] = getattr(proxy, "n_grads_used", None)
        st["grads_discarded"] = getattr(proxy, "n_grads_discarded", None)
        st["msgs_sent"] = getattr(proxy, "n_msgs_sent", None)
        st["bytes_sent"] = getattr(proxy, "bytes_sent", None)
        return st

    def _call(self, method, *args):
        rem = getattr(method, "remote", None)
        if rem is not None:
            return self.ray.get(rem(*args))
        return method(*args)

    def is_running(self) -> bool:
        return self.thread is not None and self.thread.is_alive()

    def get_error(self) -> Optional[str]:
        return self._error

    def join(self, timeout: Optional[float] = None) -> None:
        if self.thread is not None:
            self.thread.join(timeout)
        if self._error:
            raise RuntimeError(f"rank {self.rank} failed:\n{self._error}")

    def evaluate(self):
        if self.proxy is not None and hasattr(self.proxy, "quiesce"):
            self.proxy.quiesce()
        if not self._has_evaluation_callback:
            self._evaluation_callback = create_evaluation_callback(
                self.nlp, self.dev_corpus, self.T["score_weights"] or self.nlp.config["training"].get("score_weights"),
            )
            self._has_evaluation_callback = True
        return self._evaluation_callback()

    def save_checkpoint(self, info: Dict, output_path: Path) -> None:
        """Rank 0 writes the pipeline directory; every rank writes the optimizer
        state of the keys it owns (``optim/rank{r}-of{n}.pt``)."""
        output_path = Path(output_path)
        if self.proxy is not None and hasattr(self.proxy, "quiesce"):
            self.proxy.quiesce()                 # every peer's weights of the last exchange have landed
        if self.rank == 0:
            save_pipeline(self.nlp, output_path, training_cfg=self.T, info=info, before_to_disk=self.before_to_disk)
        if self.optimizer is not None and self.proxy is not None:
            master = None
            if isinstance(self.proxy, ShardedSyncProxy) and self.proxy.param_dtype != torch.float32:
                master = dict(self.proxy._master_views)
            save_optimizer_shard(output_path, self.nlp, self.optimizer, self.get_owned_keys(),
                                 rank=self.rank, world_size=self.num_workers,
                                 extra={"version": getattr(self.proxy, "version", None),
                                        "shard_balance": self._balance()},
                                 master=master)

    def _resolve_gpu(self, use_gpu: int, fused_ops: bool = True) -> int:
        if use_gpu is not None and use_gpu >= 0:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            gpu_id = int(visible.split(",")[0]) if visible.split(",")[0].strip().isdigit() else int(use_gpu)
            # Under the actor runtime each process sees exactly one device (index 0),
            # like Ray's isolation; under torchrun all devices are visible and
            # ``use_gpu`` is the local rank.
            local = 0 if ("," not in visible and visible != "") else int(use_gpu)
            assigned = os.environ.get("SRB_ASSIGNED_GPU")
            if assigned is not None:          # actor runtime: all devices visible, this one is ours
                local = gpu_id = int(assigned)
            logger.info("Using GPU (isolated): %s", gpu_id)
            require_gpu(local, fused=fused_ops)
            return gpu_id
        logger.info("Using CPU")
        require_cpu()
        return -1

    def _on_actor_shutdown(self) -> None:
        try:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


class FakeOptimizer:
    """Stand-in handed to the training loop: the real optimizer lives behind the
    proxy (``worker.py:265-278`` in the reference).  Unlike the reference's,
    ``step_schedules`` forwards to the real optimizer so learning-rate schedules
    actually advance (SURVEY.md 2.1 #7)."""

    def __init__(self, real: Any = None):
        self.averages: Dict = {}
        self._real = real

    def __call__(self, key, weights, gradient):
        return weights, gradient

    def step_schedules(self) -> None:
        if self._real is not None and hasattr(self._real, "step_schedules"):
            self._real.step_schedules()


class Evaluator:
    """Share evaluation results between workers (rank 0 publishes, others poll).
    Step-indexed: ``get_scores(i)`` returns ``None`` until the i-th evaluation has
    been published (the reference returns the *previous* scores from the second
    evaluation on, SURVEY.md 2.1 #8)."""

    def __init__(self):
        self.scores: List[Any] = []

    def set_scores(self, scores, index: Optional[int] = None):
        self.scores.append(scores)
        return scores

    def get_scores(self, index: Optional[int] = None):
        if not self.scores:
            return None
        if index is None:
            return self.scores[-1]
        return self.scores[index - 1] if len(self.scores) >= index else None


def thread_training(training_step_iterator, print_row, rank, num_workers, gpu_id, *, on_step=None, ops=None) -> None:
    if ops is not None:
        set_current_ops(ops)              # the ops selection is per-thread
    if gpu_id >= 0 and ops is not None and ops.device.type == "cuda":
        torch.cuda.set_device(ops.device)
    for batch, info, is_best_checkpoint in training_step_iterator:
        if on_step is not None:
            on_step(batch, info, is_best_checkpoint)
        if rank == 0 and is_best_checkpoint is not None:
            info = dict(info)
            info["words"] *= num_workers
            print_row(info)
