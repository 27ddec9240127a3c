"""``B200Ops``: the sm_100a backend (hand-written kernels in ``ops/csrc``).

Same interface as ``TorchOps`` (which is its numerics reference), bf16
parameters/activations, fp32 gradients.  GEMM-shaped work runs on the
tcgen05/TMEM kernels of ``gemm_tcgen05.cu`` (``use_tc=True``); with
``use_tc=False`` GEMMs go to cuBLAS via ``torch.matmul`` and only the fused
elementwise kernels are ours - that configuration is the "library GEMM"
baseline arm used to quantify what the fusion buys.

There is no silent fallback: constructing ``B200Ops`` without the built
extension raises (``python -m spacy_ray_b200.build`` builds it in-tree).

What this replaces: the reference itself ships no kernels (SURVEY.md 2.7); under
``spacy_ray/worker.py:91`` (``init_nlp``) and ``worker.py:254-262`` (``require_gpu``) it runs
thinc's ``CupyOps`` - NVRTC scalar kernels + cuBLAS fp32 - one launch per op.  Op map (SURVEY 2.7):
K1 ``multi_hash_embed*`` -> ``hash_embed_fwd_kernel`` / ``hash_embed_bwd_sorted_kernel``;
K2-K5 ``maxout_block*`` -> tcgen05 ``gemm_kernel`` (window, bias, maxout epilogue; dX from the weights
as stored; split-K dW) + ``maxout_ln_{fwd,bwd}_vec_kernel``; K6 ``softmax_xent`` -> tcgen05 logits GEMM +
``softmax_xent_bias_kernel``; K7 ``transition_steps`` -> ``biluo_block_kernel`` / ``biluo_steps_kernel`` /
``arc_eager_steps_kernel``; K8 lives in the bucketed exchange kernels (``parallel/fused_comm.py``).

Environment switches.  Defaults are the measured-fastest path; the "off" ones are complete, tested
alternatives that lost the measurement (``profiles/r2_*experiments*.md``, ``r2_fused_ln.md``):
``SRB_USE_TC``, ``SRB_TC_DW``, ``SRB_GEMM_CLUSTER`` (1 / 2 multicast / 3 pair MMA), ``SRB_GEMM_HALO``, ``SRB_DX_BN``,
``SRB_SIDE_DW``, ``SRB_SORTED_EMBED``, ``SRB_HOST_GROUP``, ``SRB_HEAD_STREAMS``, ``SRB_TAG_HEAD_TC`` (1),
``SRB_BILUO_BLOCK`` (1), ``SRB_FUSED_LN`` (0: LayerNorm in the GEMM epilogue), ``SRB_GEMM_BRES`` (0: weights
resident in shared memory), ``SRB_PDL`` / ``SRB_PDL_SIDE`` (0: programmatic dependent launch);
exchange: ``SRB_COMM_BUCKETS`` (4), ``SRB_COMM_OVERLAP``, ``SRB_COMM_PRIO``, ``SRB_NVLS`` (auto: from 4 ranks),
``SRB_GATE_ALWAYS``, ``SRB_COMM_TRACE``; engine: ``SRB_FAST_PATH*``.
"""
from __future__ import annotations

import contextlib
import os
from pathlib import Path
from typing import Any, Dict, Optional

import torch

from .torch_ops import TorchOps

_LIB = Path(__file__).parent / "_srb_cuda.so"
_loaded = False

MODE_KK, MODE_MNMN, MODE_KMN = 0, 1, 2
# what the textcat kernels hold (csrc/kernels.h kTextcat*): labels, n_pool * width, ngram_size
TEXTCAT_MAX_LABELS, TEXTCAT_MAX_POOL, TEXTCAT_MAX_NGRAM = 128, 1024, 8
EPI_STORE, EPI_MAXOUT3, EPI_ATOMIC_F32 = 0, 1, 2


def load_extension() -> None:
    global _loaded
    if _loaded:
        return
    if not _LIB.exists():
        raise RuntimeError(
            f"sm_100a extension not built: {_LIB} is missing. Run `python -m spacy_ray_b200.build` "
            "(or __graft_entry__.build()). Refusing to fall back to PyTorch ops on a GPU run."
        )
    torch.ops.load_library(str(_LIB))
    _loaded = True


def extension_available() -> bool:
    return _LIB.exists()


def _mask1d(mask: torch.Tensor) -> torch.Tensor:
    return mask.reshape(-1)


class B200Ops(TorchOps):
    name = "b200"
    fused = True
    param_dtype = torch.bfloat16

    def __init__(self, device: str = "cuda:0", *, use_tc: Optional[bool] = None, tc_dw: Optional[bool] = None):
        super().__init__(device=device, dtype=torch.bfloat16)
        if self.device.type != "cuda":
            raise ValueError("B200Ops needs a CUDA device")
        load_extension()
        self.k = torch.ops.srb
        env_tc = os.environ.get("SRB_USE_TC")
        self.use_tc = (env_tc != "0") if use_tc is None else use_tc
        env_dw = os.environ.get("SRB_TC_DW")
        self.tc_dw = (env_dw != "0") if tc_dw is None else tc_dw
        self.sorted_embed_bwd = os.environ.get("SRB_SORTED_EMBED", "1") != "0"
        # 3 = 2-CTA clusters issuing tcgen05.mma.cta_group::2 (M = 256, each CTA holds half of B);
        # 2 = 2-CTA clusters with single-CTA MMAs sharing B by TMA multicast; 1 = no clusters
        self.gemm_cluster = int(os.environ.get("SRB_GEMM_CLUSTER", "3"))
        self.dx_block_n = int(os.environ.get("SRB_DX_BN", "128"))
        self.launches = 0            # our kernels launched (bench.py reports this)
        # device-side dropout stream position: the captured training step bumps it, so CUDA-graph
        # replays draw fresh masks although the per-call seeds were baked in at capture time
        self.seed_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        # weight-gradient GEMMs that accumulate straight into the flat gradient bucket run on a side
        # stream: nothing in the backward pass reads them, and their CTAs fill the SMs the dX GEMM
        # leaves idle in its last, partial wave (201 M-tiles on 148 SMs = 1.36 waves).  The
        # consumer of the bucket (ShardedSyncProxy.step) joins the stream.
        self.side_dw = os.environ.get("SRB_SIDE_DW", "1") != "0" and self.device.type == "cuda"
        self._pdl_side = os.environ.get("SRB_PDL_SIDE", "0") == "1"
        self.tag_head_tc = os.environ.get("SRB_TAG_HEAD_TC", "1") != "0"
        # LayerNorm fused into the forward GEMM's epilogue (EPI_MAXOUT3_LN): correct and tested, but measured
        # at parity with GEMM + LayerNorm kernel (41.8 vs 41.4 us per layer, profiles/r2_fused_ln.md): off
        self.fused_ln = os.environ.get("SRB_FUSED_LN", "0") == "1"
        self._side: Optional[torch.cuda.Stream] = None
        self._side_pending = False
        self._ws: Dict[tuple, Any] = {}
        self._arc_cap: Dict[tuple, int] = {}
        self.max_rows_hint = 0               # engine.Trainer: largest row count any captured step will use
        # C2: consumer-side gates.  ``FusedSymmComm`` installs itself here; kernels that read
        # parameters ask it which buckets of freshly exchanged weights they are the first to touch
        # (``_gate``: descriptor for an in-kernel gate; ``_gate_now``: stand-alone one-warp wait in
        # front of consumers that have no in-kernel gate).
        self.gate_provider: Any = None

    def _gate(self, *tensors) -> list:
        gp = self.gate_provider
        return gp.gate_for(tensors) if gp is not None else []

    def _gate_now(self, *tensors) -> None:
        g = self._gate(*tensors)
        if g:
            self.k.gate_wait(self.gate_provider.epoch, g)
            self.launches += 1

    def side_stream_if_pending(self) -> Optional["torch.cuda.Stream"]:
        return self._side if self._side_pending else None

    # ------------------------------------------------------------------ GEMM helpers
    def _tc_ok(self, *dims: int) -> bool:
        """Dimensions the tcgen05 kernels take: multiples of 16 (UMMA N granularity; TMA needs 16-byte
        row pitches).  K need not be a multiple of the 64-element k-block and N not of the tile width:
        the TMA zero-fills what lies outside the tensor and the epilogue masks the partial last tile
        (width 96 - BASELINE config 1's model - went to cuBLAS + seq2col in round 1)."""
        return self.use_tc and all(d % 16 == 0 and d > 0 for d in dims)

    def tc_gemm(self, A, B, out, *, mode, epi, block_n, M, N, K, a_row_shift=(0,), a_col_off=(0,), b_row_off=(0,),
                b_col_off=(0,), splits=1, win_w=0, bias=None, which=None, add_src=None, row_scale=None, m_dev=None,
                max_ctas=0, cluster=None, gate=None) -> None:
        self.k.tc_gemm(A, B, out, mode, epi, block_n, M, N, K, list(a_row_shift), list(a_col_off), list(b_row_off),
                       list(b_col_off), splits, win_w, bias, which, add_src, row_scale, m_dev, max_ctas,
                       self.gemm_cluster if cluster is None else cluster, gate or [])
        self.launches += 1

    @staticmethod
    def _pick_block_n(N: int, options=(256, 192, 128, 64)) -> int:
        """Widest tile that divides N; otherwise the tile that wastes the least of a masked last tile."""
        for bn in options:
            if N % bn == 0:
                return bn
        if N % 16:
            return 0
        return min(options, key=lambda bn: (-(-N // bn) * bn, -bn))

    def _linear_tc(self, X: torch.Tensor, W: torch.Tensor, b: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        M, K = X.shape
        N = W.shape[0]
        bn = self._pick_block_n(N)
        if not (self._tc_ok(K) and bn and X.dtype == torch.bfloat16 and W.dtype == torch.bfloat16):
            return None
        out = torch.empty((M, N), dtype=torch.bfloat16, device=X.device)
        self.tc_gemm(X.contiguous(), W.contiguous(), out, mode=MODE_KK, epi=EPI_STORE, block_n=bn, M=M, N=N, K=K,
                     bias=b, gate=self._gate(W, b))
        return out

    def _dw_tc(self, dZ: torch.Tensor, X: torch.Tensor, window: int, out: Optional[torch.Tensor] = None,
               n_valid: Optional[int] = None):
        """dW[n, k] (+)= sum_t dZ[t, n] * Xw[t, k] on the tcgen05 MN-major/split-K kernel.
        ``n_valid``: only the first ``n_valid`` rows of dW exist (``dZ`` has a padded pitch whose extra
        columns are zero); ``out`` may then be the (n_valid, k) gradient buffer itself."""
        T, N = dZ.shape
        w = X.shape[1]
        if not (self.use_tc and self.tc_dw and N % 16 == 0 and w % 16 == 0):
            return None
        if window and w % 64:
            # the in-kernel window shift needs N tiles that do not straddle two shifts (64-column atoms):
            # for other widths the window is materialised once (seq2col) and the GEMM is a plain one
            X = self.k.seq2col(X.contiguous())
            self.launches += 1
            w, window = X.shape[1], 0
        Kt = w * (3 if window else 1)
        # partial tiles: a 64-row operand fills half of the 128-row M tile, the TMA zero-fills the rest
        bn = 256 if w % 256 == 0 else (128 if w % 128 == 0 else 64)
        rows = N if n_valid is None else int(n_valid)
        if out is None:
            out = torch.zeros((rows, Kt), dtype=torch.float32, device=dZ.device)
        tiles = ((rows + 127) // 128) * (Kt // bn)
        splits = max(1, min(148 // max(tiles, 1), (T + 63) // 64))
        self.tc_gemm(dZ, X, out, mode=MODE_MNMN, epi=EPI_ATOMIC_F32, block_n=bn, M=rows, N=Kt, K=T, splits=splits,
                     win_w=(w if window else 0))
        return out

    # ------------------------------------------------------------------ K1
    def multi_hash_embed(self, attrs, mask, tables, seeds, columns):
        self.launches += 1
        return self.k.hash_embed_fwd(attrs, _mask1d(mask), list(tables), list(seeds), list(columns),
                                     self._gate(*tables))

    def multi_hash_embed_backward(self, dY, attrs, mask, n_rows, seeds, columns, out=None, perm=None):
        nO = dY.shape[1] // len(n_rows)
        grads = list(out) if out is not None else [
            torch.zeros((nV, nO), dtype=torch.float32, device=dY.device) for nV in n_rows
        ]
        if self.sorted_embed_bwd:
            # sort each table's attribute column once; the kernel then reduces runs of equal
            # ids in registers and touches each table row once per run (no hot-row contention)
            cols = tuple(int(c) for c in columns)
            if perm is not None:
                # rows already grouped by id per attribute column (host counting sort shipped with
                # the batch by engine.Trainer): no device-side sort at all
                if cols != tuple(range(perm.shape[0])):
                    perm = torch.stack([perm[c] for c in cols], dim=0)
                self.k.hash_embed_bwd_sorted(dY.contiguous(), attrs, perm.contiguous(), _mask1d(mask), grads,
                                             list(seeds), list(columns))
                self.launches += 1
                return grads
            if cols == tuple(range(attrs.shape[1])):
                keys = attrs.t().contiguous()                          # (n_tables, R)
            else:                                                      # no host->device index copy (graph-safe)
                keys = torch.stack([attrs[:, c] for c in cols], dim=0).contiguous()
            # 32-bit truncated keys: half the radix passes; the kernel splits runs on the full id
            _sk, perm = torch.sort(keys.to(torch.int32), dim=1)
            self.k.hash_embed_bwd_sorted(dY.contiguous(), attrs, perm, _mask1d(mask), grads, list(seeds), list(columns))
        else:
            self.k.hash_embed_bwd(dY.contiguous(), attrs, _mask1d(mask), grads, list(seeds), list(columns))
        self.launches += 1
        return grads

    # ------------------------------------------------------------------ K2-K5
    def maxout_block(self, X, W, b, G, beta, mask, *, window=0, residual=False, dropout=0.0, is_train=False, seed=0):
        nO, nP, nI = W.shape
        Tp = X.shape[0]
        X = X.contiguous()
        W2 = W.reshape(nO * nP, nI)
        m1 = _mask1d(mask)
        drop = float(dropout) if (is_train and dropout > 0.0) else 0.0
        w_in = X.shape[1]
        use_tc = nP == 3 and self._tc_ok(w_in) and nO % 32 == 0 and window in (0, 1)
        if use_tc:
            # one tcgen05 kernel: (window) GEMM + bias + maxout; then LN/dropout/residual
            fwd_bn = 192 if nO % 64 == 0 else 96            # a tile holds all 3 pieces of 64 / 32 units
            H = torch.empty((Tp, nO), dtype=torch.bfloat16, device=X.device)
            which = torch.empty((Tp, nO), dtype=torch.uint8, device=X.device)
            if window:
                shifts = dict(a_row_shift=(-1, 0, 1), a_col_off=(0, 0, 0), b_row_off=(0, 0, 0),
                              b_col_off=(0, w_in, 2 * w_in))
            else:
                shifts = {}
            if (self.fused_ln and G is not None and fwd_bn == 192 and nO <= 512 and self.gemm_cluster == 3
                    and (not residual or w_in == nO)):
                # ONE kernel for the whole layer: the LayerNorm statistics of a row cross the N tiles as
                # two numbers per tile, the activations stay in the epilogue's registers (gemm_launch.h)
                stats, cnt = self._ln_scratch(Tp, (nO * nP) // 192)
                Y = H
                xhat = torch.empty((Tp, nO), dtype=torch.bfloat16, device=X.device)
                rstd = torch.empty((Tp,), dtype=torch.float32, device=X.device)
                sh = shifts or dict(a_row_shift=(0,), a_col_off=(0,), b_row_off=(0,), b_col_off=(0,))
                self.k.tc_gemm_maxout_ln(X, W2, Y, which, xhat, rstd, b.reshape(-1), G, beta, X if residual else None,
                                         m1, stats, cnt, Tp, nO * nP, w_in, list(sh["a_row_shift"]),
                                         list(sh["a_col_off"]), list(sh["b_row_off"]), list(sh["b_col_off"]), drop,
                                         seed, self.seed_dev, None, self.gemm_cluster, self._gate(W, b, G, beta))
                self.launches += 1
            else:
                self.tc_gemm(X, W2, H, mode=MODE_KK, epi=EPI_MAXOUT3, block_n=fwd_bn, M=Tp, N=nO * nP, K=w_in,
                             bias=b.reshape(-1), which=which, gate=self._gate(W, b, G, beta), **shifts)
                Y, _w, xhat, rstd = self.k.maxout_ln_fwd(H, None, G, beta, X if residual else None, m1, nO, 1, drop,
                                                           seed, self.seed_dev)
                self.launches += 1
        else:
            self._gate_now(W, b, G, beta)
            Xw = self.k.seq2col(X) if window else X
            Z = Xw @ W2.t()
            Y, which, xhat, rstd = self.k.maxout_ln_fwd(Z, b.reshape(-1), G, beta, X if residual else None, m1,
                                                        nO, nP, drop, seed, self.seed_dev)
            self.launches += 2 if window else 1
        ctx = {"X": X, "W": W, "which": which, "window": window, "residual": residual, "mask": m1, "nP": nP,
               "has_ln": G is not None, "xhat": xhat, "rstd": rstd, "G": G, "drop": drop, "seed": seed}
        return Y, ctx

    def _fork_side(self, *tensors: torch.Tensor) -> "torch.cuda.Stream":
        """Side stream ordered after everything issued so far on the current stream."""
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        ev = torch.cuda.Event()
        ev.record()
        self._side.wait_event(ev)
        for t in tensors:
            t.record_stream(self._side)          # the allocator must not recycle them under the side kernels
        self._side_pending = True
        return self._side

    @contextlib.contextmanager
    def _side_launches(self, *tensors: torch.Tensor):
        """Launch on the side stream.  Programmatic dependent launch (csrc/launch.h) is switched off
        for these launches: their predecessor is an event of the main stream, not the previous
        kernel of their own stream (``SRB_PDL_SIDE=1`` keeps it on)."""
        with torch.cuda.stream(self._fork_side(*tensors)):
            if self._pdl_side:
                yield
                return
            was = self.k.set_pdl(False)
            try:
                yield
            finally:
                self.k.set_pdl(was)

    def join_side(self) -> None:
        """Make the current stream wait for the side-stream gradient GEMMs (no-op if none ran)."""
        if self._side_pending:
            torch.cuda.current_stream(self.device).wait_stream(self._side)
            self._side_pending = False

    def colsum(self, X: torch.Tensor, out: Optional[torch.Tensor] = None, n_valid: Optional[int] = None) -> torch.Tensor:
        """fp32 column sums of a (T, C) bf16 matrix (bias gradients), one kernel, ACCUMULATED into
        ``out`` (which may be the gradient buffer).  ``n_valid``: only the first columns are real."""
        C = X.shape[1]
        nv = C if n_valid is None else int(n_valid)
        if out is None:
            out = torch.zeros((nv,), dtype=torch.float32, device=X.device)
        if X.dtype == torch.bfloat16 and C % 8 == 0 and C <= 2048 and X.stride(1) == 1 and X.stride(0) % 8 == 0:
            self.k.colsum_acc(X, out, nv)
            self.launches += 1
        else:
            out.add_(X[:, :nv].to(torch.float32).sum(dim=0))
        return out

    def _dx_tc(self, dY: torch.Tensor, W: torch.Tensor) -> Optional[torch.Tensor]:
        """dX = dY @ W on the tensor cores with W (nO, nI) as stored (MODE_KMN).  ``dY`` may have a
        padded pitch (K = dY.shape[1] >= W.shape[0], extra columns zero): the TMA zero-fills the
        missing rows of W, so no padded copy of the weights is made."""
        M, K = dY.shape
        N = W.shape[1]
        bn = self._pick_block_n(N)
        if not (self._tc_ok(K) and bn and dY.dtype == torch.bfloat16 and W.dtype == torch.bfloat16):
            return None
        out = torch.empty((M, N), dtype=torch.bfloat16, device=dY.device)
        self.tc_gemm(dY, W.contiguous(), out, mode=MODE_KMN, epi=EPI_STORE, block_n=bn, M=M, N=N, K=K)
        return out

    def maxout_block_backward(self, dY, ctx, grad_out: Optional[Dict[str, torch.Tensor]] = None):
        W = ctx["W"]
        nO, nP, nI = W.shape
        X = ctx["X"]
        Tp, w_in = X.shape
        window = ctx["window"]
        dev = X.device
        has_ln = ctx["has_ln"]
        # ``grad_out``: fp32 views of the flat gradient bucket.  Kernels accumulate straight into
        # them (atomics / split-K red), so no zero-fill + add_ launches per parameter.
        go = grad_out or {}

        def _dst(name, shape):
            t = go.get(name)
            if t is not None and t.dtype == torch.float32 and t.is_contiguous():
                return t.view(shape)
            return torch.zeros(shape, dtype=torch.float32, device=dev)

        db = _dst("b", (nO * nP,))
        dG = _dst("G", (nO,)) if has_ln else None
        dbeta = _dst("beta", (nO,)) if has_ln else None
        dY = dY.contiguous()
        dZ = self.k.maxout_ln_bwd(dY, ctx["xhat"] if has_ln else None, ctx["rstd"] if has_ln else None,
                                  ctx["G"], ctx["which"], ctx["mask"], nP, ctx["drop"], ctx["seed"], db, dG, dbeta,
                                  self.seed_dev)
        self.launches += 1
        W2 = W.reshape(nO * nP, nI)
        N = nO * nP
        # ---- dW ----------------------------------------------------------
        dW_dst = go.get("W")
        if dW_dst is not None and not (dW_dst.dtype == torch.float32 and dW_dst.is_contiguous()):
            dW_dst = None
        if dW_dst is not None and self.side_dw and self.use_tc and self.tc_dw:
            with self._side_launches(dZ, X):
                dW = self._dw_tc(dZ, X, window, out=dW_dst.view(nO * nP, nI))
            if dW is None:
                self.join_side()
        else:
            dW = self._dw_tc(dZ, X, window, out=dW_dst.view(nO * nP, nI) if dW_dst is not None else None)
        if dW is None:
            Xw = self.k.seq2col(X) if window else X
            dW = _mm_f32(dZ.t(), Xw)
            if dW_dst is not None:
                dW_dst.view(nO * nP, nI).add_(dW)
                dW = dW_dst
        # ---- dX ----------------------------------------------------------
        bn = self._pick_block_n(w_in)
        if window and bn and w_in % self.dx_block_n == 0:
            # halo window GEMM: 128-wide N tiles give a 4-stage ring and 2.7 waves instead of 3 stages /
            # 1.36 waves (measured 34.4 vs 41.8 us at the flagship shape)
            bn = self.dx_block_n
        if self._tc_ok(N, w_in) and bn:
            # B = the weights as stored, (N, nI) = (K, N) row-major -> MN-major UMMA operand: no
            # per-step transpose of W (it changes every step, so a cached W^T is useless)
            W2c = W2.contiguous()
            dX = torch.empty((Tp, w_in), dtype=torch.bfloat16, device=dev)
            if window:
                self.tc_gemm(dZ, W2c, dX, mode=MODE_KMN, epi=EPI_STORE, block_n=bn, M=Tp, N=w_in, K=N,
                             a_row_shift=(1, 0, -1), a_col_off=(0, 0, 0), b_row_off=(0, 0, 0),
                             b_col_off=(0, w_in, 2 * w_in), add_src=dY if ctx["residual"] else None,
                             row_scale=ctx["mask"] if ctx["residual"] else None)
            else:
                self.tc_gemm(dZ, W2c, dX, mode=MODE_KMN, epi=EPI_STORE, block_n=bn, M=Tp, N=w_in, K=N,
                             add_src=dY if ctx["residual"] else None,
                             row_scale=ctx["mask"] if ctx["residual"] else None)
        else:
            dXw = dZ @ W2
            if window:
                dX = self.k.col2seq_residual(dXw, dY if ctx["residual"] else None, ctx["mask"])
                self.launches += 1
            else:
                dX = dXw + dY * ctx["mask"].unsqueeze(1).to(dY.dtype) if ctx["residual"] else dXw
        return dX, dW.view(nO, nP, nI), db.view(nO, nP), dG, dbeta

    # ------------------------------------------------------------------ Linear
    def linear(self, X, W, b):
        X = X.contiguous()
        if X.dtype != torch.bfloat16:
            X = X.to(torch.bfloat16)
        out = self._linear_tc(X, W, b)
        if out is not None:
            return out
        self._gate_now(W, b)
        Y = X @ W.t()
        return Y + b if b is not None else Y

    def linear_backward(self, dY, X, W, need_dX: bool = True, need_db: bool = True,
                        grad_out: Optional[Dict[str, torch.Tensor]] = None):
        """``grad_out``: fp32 views of the flat gradient bucket for ``W`` / ``b``; the split-K GEMM and
        the column-sum kernel accumulate straight into them (no zero-fill + add launches)."""
        dY = dY.to(torch.bfloat16).contiguous() if dY.dtype != torch.bfloat16 else dY.contiguous()
        X = X.contiguous()
        go = grad_out or {}
        gW, gb = go.get("W"), go.get("b")
        if gW is not None and not (gW.dtype == torch.float32 and gW.is_contiguous()):
            gW = None
        if gb is not None and not (gb.dtype == torch.float32 and gb.is_contiguous()):
            gb = None
        dW = self._dw_tc(dY, X, 0, out=gW.view(W.shape) if gW is not None else None)
        if dW is None:
            dW = _mm_f32(dY.t(), X)
            if gW is not None:
                gW.view(W.shape).add_(dW)
                dW = gW
        db = self.colsum(dY, out=gb.view(-1) if gb is not None else None) if need_db else None
        dX = None
        if need_dX:
            dX = self._dx_tc(dY, W)
            if dX is None:
                dX = dY @ W
        return dX, dW, db

    # ------------------------------------------------------------------ K6
    def softmax(self, logits):
        return torch.softmax(logits.to(torch.float32), dim=-1)

    def softmax_xent(self, X, W, b, labels, grad_out: Optional[Dict[str, torch.Tensor]] = None):
        self._gate_now(W, b)
        X = X.contiguous()
        nC = W.shape[0]
        if X.dtype == torch.bfloat16 and W.dtype == torch.bfloat16 and X.shape[1] % 16 == 0 and nC <= 128:
            out = None
            if self.use_tc and self.tag_head_tc:
                # K6 on the tensor cores: logits = X W^T accumulated into a persistent zeroed fp32 scratch by the
                # tcgen05 GEMM (rows of W past nC are zero-filled by the TMA), then ONE kernel for bias + softmax +
                # CE gradient + loss + argmax, which also leaves the scratch zeroed for the next step
                T, w = X.shape
                n16 = (nC + 15) // 16 * 16
                bn = 64 if n16 <= 64 else 128
                # (one scratch per head - keyed by its weights - because the heads of a multi-task pipeline run
                # on concurrent streams; allocated by the eager first step, never under capture)
                logits = self._workspace(f"tag_logits@{W.data_ptr():x}", T, bn)
                self.tc_gemm(X, W.contiguous(), logits, mode=MODE_KK, epi=EPI_ATOMIC_F32, block_n=bn, M=T, N=n16, K=w,
                             splits=1, cluster=1)
                out = self.k.softmax_xent_bias(logits, b.to(torch.bfloat16).contiguous(), labels.contiguous(), nC)
            else:
                # K6 in one CUDA-core kernel (W in shared memory): fine for narrow models only
                out = self.k.linear_softmax_xent(X, W.contiguous(), b.to(torch.bfloat16).contiguous(),
                                                 labels.contiguous())
            if out:
                dp, guesses, loss = out                        # dp: (T, 128k) bf16, zero past nC
                self.launches += 1
                gW, gb = (grad_out or {}).get("W"), (grad_out or {}).get("b")
                if gW is not None and not (gW.dtype == torch.float32 and gW.is_contiguous()):
                    gW = None
                if gb is not None and not (gb.dtype == torch.float32 and gb.is_contiguous()):
                    gb = None
                dW = self._dw_tc(dp, X, 0, out=gW.view(W.shape) if gW is not None else None, n_valid=nC)
                if dW is None:
                    dW = _mm_f32(dp[:, :nC].t(), X)
                    if gW is not None:
                        gW.view(W.shape).add_(dW)
                        dW = gW
                db = self.colsum(dp, out=gb.view(-1) if gb is not None else None, n_valid=nC)
                dX = self._dx_tc(dp, W)                           # rows >= nC of W: zero-filled by the TMA
                if dX is None:
                    dX = dp[:, :nC] @ W
                return loss, dp[:, :nC], guesses, dX, dW, db
        logits = (X @ W.t()).to(torch.float32) + b.to(torch.float32)
        d, guesses, loss = self.k.softmax_xent(logits.contiguous(), labels.contiguous())
        self.launches += 1
        dW = _mm_f32(d.t(), X)
        db = self.colsum(d)
        dX = d @ W
        return loss, d, guesses, dX, dW, db

    # ------------------------------------------------------------------ textcat head
    def textcat_head(self, X, batch, W, b, W_bow, b_bow, truths, known, *, n_docs=None, use_mean: bool = True,
                     use_max: bool = False, exclusive: bool = True, no_output_layer: bool = False,
                     ngram_size: int = 1, grad_out: Optional[Dict[str, torch.Tensor]] = None):
        """``TorchOps.textcat_head`` in two kernels (textcat_kernels.cu): one CTA per doc for pooling, the
        bag of n-grams, the output layer, the loss, dX and the W_bow gradient rows; one reduction over docs
        for dW / db / the loss.  ``n_docs`` may be a device int32 tensor (the engine's packed buffer), so
        nothing here reads the host.  Gradients accumulate straight into ``grad_out`` (fp32 views of the
        flat bucket) when given."""
        weights = [t for t in (W, b, W_bow, b_bow) if t is not None]
        self._gate_now(*weights)
        dev = truths.device
        nL = int(truths.shape[1])
        go = {k: v for k, v in (grad_out or {}).items()
              if v is not None and v.dtype == torch.float32 and v.is_contiguous()}
        grads: Dict[str, torch.Tensor] = {}
        for name, p in (("W", W), ("b", b), ("W_bow", W_bow), ("b_bow", b_bow)):
            if p is not None:
                grads[name] = go[name].view(p.shape) if name in go else torch.zeros(p.shape, dtype=torch.float32,
                                                                                     device=dev)
        n_dev, n_host = None, int(batch.doc_lens.numel())
        if isinstance(n_docs, torch.Tensor):
            n_dev = n_docs.reshape(-1)[:1]
        elif n_docs is not None:
            n_host = int(n_docs)
        act = 2 if no_output_layer else (0 if exclusive else 1)
        Xc = X.contiguous() if X is not None else None
        loss, scores, dX, _pooled, _dl = self.k.textcat_head(
            Xc, _mask1d(batch.mask).to(torch.float32).contiguous(), batch.attrs.contiguous(), batch.doc_starts,
            batch.doc_lens, n_dev, n_host, W.contiguous() if W is not None else None,
            b.contiguous() if b is not None else None, W_bow.contiguous() if W_bow is not None else None,
            b_bow.contiguous() if b_bow is not None else None, truths.contiguous(), known.contiguous(),
            grads.get("W"), grads.get("b"), grads.get("W_bow"), grads.get("b_bow"), nL, bool(use_mean),
            bool(use_max), act, int(ngram_size))
        self.launches += 2
        return loss, scores, (dX if X is not None else None), grads

    # ------------------------------------------------------------------ K7
    def transition_steps(self, system, Yf, params, batch, gold, is_train):
        from ..models.transitions import ArcEagerSystem, BiluoSystem

        self._gate_now(params["pad"], params["b"], params["Wu"], params["bu"])
        if isinstance(system, ArcEagerSystem):
            return self._arc_eager_steps(system, Yf, params, batch, gold, is_train)
        if not isinstance(system, BiluoSystem):
            return None
        nO, nP = params["nO"], params["nP"]
        if nP != 2 or nO % 32 != 0 or (nO * nP) // 32 > 8 or system.n_actions > 256:
            return None
        dev = Yf.device
        extra = batch.extra
        tok_off = extra.get("tok_off")
        if tok_off is None:
            lens = batch.doc_lens.to(torch.int64)
            tok_off = (torch.cumsum(lens, 0) - lens).to(torch.int32)
            extra["tok_off"] = tok_off
        inv_active = extra.get("inv_active")
        if inv_active is None:
            max_len = max(batch.lengths) if batch.lengths else 1
            lens_t = torch.tensor(batch.lengths, dtype=torch.int64)
            counts = (lens_t.unsqueeze(0) > torch.arange(max_len).unsqueeze(1)).sum(dim=1).clamp(min=1)
            inv_active = (1.0 / counts.to(torch.float32)).to(dev)
            extra["inv_active"] = inv_active
        gold_t = None
        if is_train and gold is not None and gold.actions is not None:
            gold_t = gold.actions.to(torch.int32)
        feats, which, hid, d_scores, actions, loss = self.k.biluo_steps(
            Yf.contiguous(), params["pad"].contiguous(), params["b"].contiguous(), params["Wu"].contiguous(),
            params["bu"].contiguous(), batch.doc_starts, batch.doc_lens, tok_off, gold_t, inv_active,
            batch.n_tokens, nO, nP, system.n_labels, bool(is_train and gold_t is not None),
            bool(getattr(gold, "teacher_forced", False)),
        )
        self.launches += 1
        rec: Dict[str, Any] = {"actions_flat": actions, "loss": loss, "n_steps": 0}      # int32
        if is_train and gold_t is not None:
            rec.update({"feats": feats, "which": which, "hid": hid, "d_scores": d_scores,
                        "n_steps": batch.n_tokens, "nA": system.n_actions})
        return rec

    def _arc_eager_steps(self, system, Yf, params, batch, gold, is_train):
        """Arc-eager derivations of the whole batch in one kernel (parser_kernels.cu)."""
        import numpy as np

        from ..nn.batch import to_device

        nO, nP = params["nO"], params["nP"]
        # longest doc of the batch: host-side lengths, or the engine's staging capacity
        max_len = max(batch.lengths) if batch.lengths else int(batch.extra.get("max_len", 128))
        if nO % 32 != 0 or nO // 32 not in (1, 2, 4) or nP not in (2, 3) or system.n_actions > 192:
            return None                       # host state machine (reference loop)
        if max_len > self.arc_eager_capacity(nO, nP, system.n_actions):
            return None                       # the per-warp parser state would not fit in shared memory
        dev = Yf.device
        extra = batch.extra
        if "tok_off" not in extra:
            lens = batch.doc_lens.to(torch.int64)
            extra["tok_off"] = (torch.cumsum(lens, 0) - lens).to(torch.int32)
        if "step_off" not in extra:
            extra["step_off"] = (extra["tok_off"] * 2).to(torch.int32)
        train = bool(is_train and gold is not None and (gold.heads is not None or gold.heads_flat is not None))
        gh = gl = None
        if train:
            gh, gl = gold.heads_flat, gold.labels_flat
            if gh is None:
                gh = to_device(np.asarray([h for doc in gold.heads for h in doc], dtype=np.int32), dev)
                gl = to_device(np.asarray([l for doc in gold.labels for l in doc], dtype=np.int32), dev)
        S_cap = 2 * batch.n_tokens
        feats, which, hid, d_scores, history, heads, labels, n_steps, loss = self.k.arc_eager_steps(
            Yf.contiguous(), params["pad"].contiguous(), params["b"].contiguous(), params["Wu"].contiguous(),
            params["bu"].contiguous(), batch.doc_starts, batch.doc_lens, extra["tok_off"], extra["step_off"],
            gh, gl, batch.n_tokens, S_cap, nO, nP, 1.0 / max(1, batch.n_docs), train,
            bool(getattr(gold, "teacher_forced", False)), int(max(max_len, 1)),
        )
        self.launches += 1
        rec: Dict[str, Any] = {"arc_heads": heads, "arc_labels": labels, "loss": loss, "n_steps": 0,
                               "arc_history": history, "arc_n_steps": n_steps}
        if train:
            rec.update({"feats": feats, "which": which, "hid": hid, "d_scores": d_scores, "n_steps": S_cap,
                        "nA": system.n_actions})
        return rec

    def _ln_scratch(self, rows: int, n_tiles: int):
        """Scratch of the fused LayerNorm epilogue (csrc/gemm_launch.h): the tagged per-row partial sums
        (fp32, zeroed once) and the kernel-maintained [launch tag, finished CTAs, time-out flag] words.
        Persistent and sized once like ``_workspace`` (``max_rows_hint``)."""
        need = (rows + 255) // 256 * 256
        # (one scratch per width class, allocated by the eager first step - never under capture; the fused
        # epilogue therefore assumes the encoders of a pipeline run on ONE stream, which is how the engine
        # schedules a shared tok2vec)
        key = ("ln_scratch", n_tiles)
        cur = self._ws.get(key)
        if cur is None or cur[2] < need:
            rows_pad = (max(rows, int(self.max_rows_hint)) + 255) // 256 * 256
            stats = torch.zeros((rows_pad * n_tiles * 4,), dtype=torch.float32, device=self.device)
            seq = torch.tensor([1, 0, 0], dtype=torch.int32, device=self.device)
            cur = self._ws[key] = (stats, seq, rows_pad)
        return cur[0], cur[1]

    def check_fused_ln(self) -> None:
        """Raise if a fused-LayerNorm epilogue ever timed out waiting for another tile's statistics."""
        for key, cur in self._ws.items():
            if key[0] == "ln_scratch" and int(cur[1][2].item()) != 0:
                raise RuntimeError("fused LayerNorm epilogue: a wait on the row statistics timed out")

    def _workspace(self, name: str, rows: int, cols: int) -> torch.Tensor:
        """Persistent zero-initialised fp32 scratch, (>= rows, cols): allocated once (at the largest row
        count the engine announced via ``max_rows_hint``) and handed out as a row slice, so captured
        steps neither allocate nor memset it - its users leave it zeroed."""
        key = (name, cols)
        ws = self._ws.get(key)
        if ws is None or ws.shape[0] < rows:
            ws = self._ws[key] = torch.zeros((max(rows, int(self.max_rows_hint)), cols), dtype=torch.float32,
                                             device=self.device)
        return ws[:rows]

    def arc_eager_capacity(self, nO: int, nP: int, n_actions: int) -> int:
        """Longest doc (tokens) the device arc-eager kernel handles for this head shape."""
        key = (nO, nP, n_actions)
        cap = self._arc_cap.get(key)
        if cap is None:
            cap = self._arc_cap[key] = int(self.k.arc_eager_capacity(nO, nP, n_actions))
        return cap

    def transition_backward(self, rec, params, n_rows, grad_out: Optional[Dict[str, torch.Tensor]] = None):
        if rec["d_scores"].dtype != torch.bfloat16:
            return None                       # records from the reference loop: use the reference backward
        nF, nO, nP = params["nF"], params["nO"], params["nP"]
        nA = rec["nA"]
        d = rec["d_scores"]                   # (S, nA_pad) bf16, padded columns are zero
        hid = rec["hid"]
        dev = d.device
        go = {k: v for k, v in (grad_out or {}).items()
              if v is not None and v.dtype == torch.float32 and v.is_contiguous()}
        # d has a 128-multiple pitch (zero columns past nA), so both products run on the tcgen05 kernels;
        # only the nA real rows / columns are written, straight into the gradient bucket when given
        gWu = go.get("Wu")
        dWu = self._dw_tc(d, hid, 0, out=gWu.view(nA, nO) if gWu is not None else None, n_valid=nA)
        if dWu is None:
            dWu = _mm_f32(d[:, :nA].t(), hid)
            if gWu is not None:
                gWu.view(nA, nO).add_(dWu)
                dWu = gWu
        dbu = self.colsum(d, out=go["bu"].view(-1) if "bu" in go else None, n_valid=nA)
        d_hid = self._dx_tc(d, params["Wu"])                 # rows >= nA of Wu: zero-filled by the TMA
        if d_hid is None:
            d_hid = (d[:, :nA] @ params["Wu"]).contiguous()
        dYf32 = self._workspace("dYf", n_rows, nF * nO * nP)
        dpad = go["pad"].view(nF, nO * nP) if "pad" in go else torch.zeros((nF, nO * nP), dtype=torch.float32, device=dev)
        db = go["b"].view(nO * nP) if "b" in go else torch.zeros((nO * nP,), dtype=torch.float32, device=dev)
        self.k.transition_scatter(d_hid, rec["which"], rec["feats"], dYf32, dpad, db, nF, nP)
        dYf = self.k.f32_to_bf16_zero(dYf32)                 # bf16 for the GEMMs below; the scratch is clear again
        self.launches += 2
        return {"dWu": dWu, "dbu": dbu, "db": db, "dpad": dpad, "dYf": dYf}

    # ------------------------------------------------------------------ misc
    def gemm(self, A, B, trans1=False, trans2=False):
        self._gate_now(A, B)
        a = A.t() if trans1 else A
        b = B.t() if trans2 else B
        return a.to(torch.bfloat16) @ b.to(torch.bfloat16)


def _mm_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """bf16 x bf16 -> fp32 output (cuBLAS accumulates in fp32 either way)."""
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except (TypeError, RuntimeError):
        return (a.to(torch.float32) @ b.to(torch.float32))
