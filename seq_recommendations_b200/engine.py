"""Device-side orchestration of the hot path: one `HotPath` object owns the weights, gradients, optimizer state and
work buffers in HBM and sequences the C-ABI kernels (include/seqrec_b200.h) on the current CUDA stream.

What it replaces in the reference: everything Keras/Theano executes under `self.model.fit(...)`,
`self.model.evaluate(...)` and `self.model.predict(...)` (model.py:181, :195, :198) for the recurrent models
(model.py:241-258, :322-403) trained with Adagrad + clipnorm (experiments_methods.py:41-42).

PyTorch is plumbing here (device memory, streams, NCCL); every arithmetic step of the path is a kernel of
libseqrec_b200.so.  There is no CPU path: constructing a HotPath without CUDA or without the library raises.

HBM layout (all fp32 unless noted; token n = t*B + b, time-major):
  weights   W_in (F,G*H) | flat[U (H,G*H) | b (G*H) | W_out (H,V) | b_out (V)]         Keras layouts, row-major
  grads     ONE allocation: dW_in (F,G*H) zero-invariant | step floats [n_valid, loss_sum, ...] | flat like the weights |
            per-step integer scalars (n_valid, touched-row count, squared gradient norm).  One fill clears everything
            behind dW_in at the start of a step; one all-reduce covers [dW_in |] step floats | dU | db.  Gradients are
            stored UN-normalised (sums over tokens); the optimiser kernels divide by the global n_valid
  accum     Adagrad accumulators, same shapes -- or Adam's second moments v, with the first moments m in buffers of
            the same shapes allocated when Adam is selected, and the update count `iterations` (device int64)
  per batch ids/tgt int32 [T][B], mask u8 [T][B], xg [T][B][G*H] (xp -> gates -> dxp in place),
            hout [T][B][H], cst [T][B][H], dh [T][B][H], per-token stats m,s,zy,ce,py,coef [N], ws [splits][N]
"""
import contextlib
import ctypes
import gc
import math
import os

import numpy as np
import torch

from . import _lib
from ._lib import ACT, CELL, call, ptr
from .dist import Comm, embedding_grad_mode
from .gemm import gemm
from .ranking import check_candidates
from .state import RecurrentState

GATES = {"simpleRNN": 1, "LSTM": 4, "GRU": 3}
NUM_SMS = 148


def _align(n, a=64):
    return (n + a - 1) // a * a


def _optimizer_spec(kind, lr, epsilon, clipnorm, decay, beta_1, beta_2):
    """HotPath.opt / DensePath.opt: the hyper-parameters of Adagrad or Keras Adam."""
    if kind not in ("adagrad", "adam"):
        raise NotImplementedError("optimizer %r: Adagrad (the reference's, experiments_methods.py:41) and Adam are "
                                  "built" % (kind,))
    if kind == "adagrad" and decay:
        raise NotImplementedError("learning-rate decay is never used by the reference (decay=0.0)")
    if kind == "adam" and not (0.0 <= beta_1 < 1.0 and 0.0 <= beta_2 < 1.0 and decay >= 0.0):
        raise ValueError("Adam needs 0 <= beta_1, beta_2 < 1 and decay >= 0")
    return dict(kind=kind, lr=float(lr), eps=float(epsilon), clipnorm=float(clipnorm or 0.0), decay=float(decay or 0.0),
                beta_1=float(beta_1), beta_2=float(beta_2))


class _Work:
    """Per-(B,T) work buffers."""

    def __init__(self, hp, B, T):
        dev = hp.device
        N = B * T
        f32, i32 = torch.float32, torch.int32
        self.B, self.T, self.N = B, T, N
        self.ids_bt = torch.empty((B, T), dtype=i32, device=dev)
        self.tgt_bt = torch.empty((B, T), dtype=i32, device=dev)
        self.ids = torch.empty((T, B), dtype=i32, device=dev)
        self.tgt = torch.empty((T, B), dtype=i32, device=dev)
        self.mask = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.n_valid_i = hp.scal[0:1]               # shared per-step scalar block (HotPath.scal)
        self.loss_mean = torch.zeros(1, dtype=f32, device=dev)
        self.xg = torch.empty((T, B, hp.GH), dtype=f32, device=dev)
        self.hout = torch.empty((T, B, hp.H), dtype=f32, device=dev)
        self.cst = torch.empty((T, B, hp.H), dtype=f32, device=dev)
        self.dh = torch.empty((T, B, hp.H), dtype=f32, device=dev)
        self.splits = hp._ce_splits(N)
        self.ws_m = torch.empty((self.splits, N), dtype=f32, device=dev)
        self.ws_s = torch.empty((self.splits, N), dtype=f32, device=dev)
        self.m = torch.empty(N, dtype=f32, device=dev)
        self.s = torch.empty(N, dtype=f32, device=dev)
        self.zy = torch.zeros(N, dtype=f32, device=dev)
        self.ce = torch.empty(N, dtype=f32, device=dev)
        self.py = torch.empty(N, dtype=f32, device=dev)
        self.coef = torch.empty(N, dtype=f32, device=dev)
        self.loss_sum = torch.zeros(1, dtype=f32, device=dev)
        self.hscale = None
        self.in_scale = None
        self.rec_mask = None
        self.rd_scratch = None
        self.orig = self.tgt_c = self.n_c = self.blk = self.acc = self.ce_tgt = self.ce_n = None
        self.pz = self.pz_hi = self.pz_lo = self.pzt_hi = self.pzt_lo = None
        self.x_dense = None
        self.pin_event = None
        self.pin_dirty = False
        self.graph = None
        self.graph_key = None
        self.graph_calls = 0
        self.graph_loss = None
        self.D_hi = self.D_lo = self.Hs_hi = self.Hs_lo = self.C_hi = self.C_lo = None   # bf16 operands of the dU GEMM
        self.tc_operands_fresh = False         # A_hi / A_lo hold the split of the CURRENT hout
        # bf16 hi/lo operands of the tensor-core logits kernels (zero padding of Hk / Np is never written)
        self.tc = hp._tc_plan(N)
        if self.tc["fwd"] or self.tc["panel_tc"]:
            bf = torch.bfloat16
            self.Np = (N + 7) // 8 * 8
            self.A_hi = torch.zeros((N, hp.Hk), dtype=bf, device=dev)
            self.A_lo = torch.zeros((N, hp.Hk), dtype=bf, device=dev) if hp.tc_x3 else None
            if self.tc["bwd"] or self.tc["panel_tc"]:
                self.Ht_hi = torch.zeros((hp.Hk, self.Np), dtype=bf, device=dev)
                self.Ht_lo = torch.zeros((hp.Hk, self.Np), dtype=bf, device=dev) if hp.tc_x3 else None
            if self.tc["splits"] > self.splits:
                self.splits = self.tc["splits"]
                self.ws_m = torch.empty((self.splits, N), dtype=f32, device=dev)
                self.ws_s = torch.empty((self.splits, N), dtype=f32, device=dev)
        # pinned staging for host batches
        self.pin_ids = torch.empty((B, T), dtype=i32, pin_memory=True)
        self.pin_tgt = torch.empty((B, T), dtype=i32, pin_memory=True)


class HotPath:
    def __init__(self, cell, act, in_dim, hidden, n_items, out_bias=False, input_kind="ids", weights=None,
                 device=None, comm=None, seed=0, tc="x3", vocab_parallel=False):
        if not torch.cuda.is_available():
            raise _lib.SeqrecError("seq_recommendations_b200 needs a CUDA device (sm_100a); there is no CPU path")
        _lib.load()
        if cell not in CELL:
            raise ValueError("rnn_type must be one of %s" % sorted(CELL))
        if act not in ACT:
            raise ValueError("activation must be one of %s" % sorted(ACT))
        if input_kind not in ("ids", "dense"):
            raise ValueError(input_kind)
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.cell, self.act = cell, act
        self.G = GATES[cell]
        self.F, self.H, self.V = int(in_dim), int(hidden), int(n_items)
        self.GH = self.G * self.H
        self.out_bias = bool(out_bias)
        self.input_kind = input_kind
        self.comm = comm if comm is not None else Comm()
        # Vocabulary-parallel logits (SURVEY §8(e), large catalogs): W_out / b_out are column-sharded, every rank
        # scores ALL ranks' tokens against its V/P items; the recurrent part stays data parallel.  self.V is the
        # LOCAL item count from here on, self.V_total the catalog size, self.v_lo the first local item.
        self.V_total = self.V
        self.v_lo = 0
        self.vocab_parallel = bool(vocab_parallel) and self.comm.enabled
        if self.vocab_parallel:
            if self.V_total % self.comm.world:
                raise ValueError("vocab_parallel needs n_items divisible by the number of ranks")
            self.V = self.V_total // self.comm.world
            self.v_lo = self.comm.rank * self.V
        self.dropout_in = 0.0
        self.dropout_out = 0.0
        self.dropout_rec = 0.0                     # Keras recurrent_dropout (z -> z), model.py:346,351
        # identical seeds on every rank would draw identical dropout masks for different shards: fold the rank in
        self.seed = int(seed) * max(1, self.comm.world) + self.comm.rank
        # dropout stream position, on the device ([0] next offset, [1] kernel-internal ticket): a captured step draws
        # fresh factors at every replay
        self.rng_state = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._work = {}
        f32 = torch.float32
        dev = self.device
        # flat parameter / gradient / accumulator buffers: U | b | W_out | b_out (64-float aligned segments)
        sizes = [self.H * self.GH, self.GH, self.H * self.V, self.V if self.out_bias else 0]
        offs, o = [], 0
        for s in sizes:
            offs.append(o)
            o += _align(s)
        self._seg = list(zip(offs, sizes))
        self.flat_p = torch.zeros(o, dtype=f32, device=dev)
        # ONE gradient allocation: dW_in (zero-invariant: only touched rows are ever non-zero, the row-sparse Adagrad
        # re-zeroes them) | 64 step floats | flat dense gradients | 4 words of integer step scalars.  A training step
        # clears everything behind dW_in with ONE fill when the batch is staged; a data-parallel step reduces
        # [dW_in (dense exchange only) | step floats | dU | db] in ONE all-reduce.
        #   stepf[0] unmasked tokens (float), [1] loss sum, [2] squared norm of the vocabulary-sharded gradients
        #   scal[0] unmasked tokens (int32), [1] touched-row count (int32), [2:4] squared gradient norm (float64)
        self._fgh = _align(self.F * self.GH)
        self._gbuf = torch.zeros(self._fgh + 64 + o + 4, dtype=f32, device=dev)
        self.dW_in = self._gbuf[:self.F * self.GH].view(self.F, self.GH)
        self.stepf = self._gbuf[self._fgh:self._fgh + 64]
        self._grads_and_scal = self._gbuf[self._fgh:]
        self.flat_g = self._gbuf[self._fgh + 64:self._fgh + 64 + o]
        self.scal = self._gbuf[self._fgh + 64 + o:].view(torch.int32)
        self.flat_a = torch.zeros(o, dtype=f32, device=dev)
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=dev)   # id range violations seen by format_batch

        def views(flat):
            U = flat[offs[0]:offs[0] + sizes[0]].view(self.H, self.GH)
            b = flat[offs[1]:offs[1] + sizes[1]]
            Wo = flat[offs[2]:offs[2] + sizes[2]].view(self.H, self.V)
            bo = flat[offs[3]:offs[3] + sizes[3]] if self.out_bias else None
            return U, b, Wo, bo

        self.U, self.b, self.W_out, self.b_out = views(self.flat_p)
        self.dU, self.db, self.dW_out, self.db_out = views(self.flat_g)
        self.aU, self.ab, self.aW_out, self.ab_out = views(self.flat_a)      # Adagrad accumulators / Adam's v
        self._views = views
        self.W_in = torch.zeros((self.F, self.GH), dtype=f32, device=dev)
        self.aW_in = torch.zeros((self.F, self.GH), dtype=f32, device=dev)
        # Adam's first moments (flat_m, mW_in and the m* views): allocated when Adam is first selected, then kept, so a
        # captured step's pointers stay valid.  iterations = updates applied so far, read by the Adam kernels.
        self.flat_m = self.mU = self.mb = self.mW_out = self.mb_out = self.mW_in = None
        self.iterations = torch.zeros(1, dtype=torch.int64, device=dev)
        self.Ut = torch.empty((self.GH, self.H), dtype=f32, device=dev)
        self._needs_ut = _lib.load().seqrec_rnn_needs_ut(CELL[cell], self.H) != 0
        # tensor-core recurrent scan (csrc/rnn_tc.cu): LSTM / GRU with H in {128, 256}.  The register-resident SIMT scan
        # stays the default for GRU-128 (2 us per step already); SEQREC_RNN_TC=1 / 0 forces / disables it.
        lib = _lib.load()
        tc_ok = lib.seqrec_rnn_tc_applicable(CELL[cell], self.H) != 0
        env = os.environ.get("SEQREC_RNN_TC", "")
        self.Ut_hi = self.Ut_lo = self.U_hi = self.U_lo = None
        # recurrent weight gradient as a split-K tcgen05 GEMM over all tokens (csrc/wgrad_tc.cu); SEQREC_WGRAD_TC=0 disables
        self.wgrad_tc = tc_ok and os.environ.get("SEQREC_WGRAD_TC", "1") != "0"
        self.rnn_tc = tc_ok and (env == "1" or (env != "0" and (self.H > 128 or cell == "LSTM")))
        if tc_ok:
            self.Ut_hi = torch.empty((self.GH, self.H), dtype=torch.bfloat16, device=dev)
            self.Ut_lo = torch.empty((self.GH, self.H), dtype=torch.bfloat16, device=dev)
            self.U_hi = torch.empty((self.H, self.GH), dtype=torch.bfloat16, device=dev)
            self.U_lo = torch.empty((self.H, self.GH), dtype=torch.bfloat16, device=dev)
        self.touched = torch.zeros(self.F, dtype=torch.int32, device=dev)
        self.rows = torch.empty(self.F, dtype=torch.int32, device=dev)
        self.n_rows = self.scal[1:2]
        self.sumsq = self.scal[2:4].view(torch.float64)
        self.n_valid_f = self.stepf[0:1]
        self.step_loss_sum = self.stepf[1:2]
        self.trainable = {"W_in": True, "U": True, "b": True, "W_out": True, "b_out": True}
        self.opt = None
        self.prof = None  # list of (phase name, cuda event) marks when bench.py profiles a step
        self.use_graphs = os.environ.get("SEQREC_GRAPHS", "1") == "1"
        # independent short kernels of a step (operand staging | scan, target logit | logits pass, scatter-add | dU
        # GEMMs, dense | row-sparse optimiser halves) run as parallel branches: a second stream, forked and joined with
        # events -- under CUDA-graph capture these become parallel branches of the step graph
        self.overlap = os.environ.get("SEQREC_OVERLAP", "1") == "1"
        self._side_stream = torch.cuda.Stream(device=dev) if dev.type == "cuda" else None
        self.graph_collectives = os.environ.get("SEQREC_GRAPH_COLLECTIVES", "1") == "1"   # capture NCCL calls too
        # tensor-core logits path: 'x3' = 3-pass bf16 split products (fp32-grade, the default), 'bf16' = single pass,
        # 'off' = exact-fp32 SIMT kernels.  SEQREC_TC overrides.  Small / odd problems always take the SIMT kernels.
        self.tc_mode = os.environ.get("SEQREC_TC", tc)
        if self.tc_mode not in ("x3", "bf16", "off"):
            raise ValueError("tc must be 'x3', 'bf16' or 'off'")
        self.tc_x3 = self.tc_mode == "x3"
        # training: forward statistics and dH from ONE logits pass (seqrec_ce_tc_fused); SEQREC_CE_FUSED=0 falls back to
        # the separate forward + token-stationary backward kernels
        self.ce_fused = os.environ.get("SEQREC_CE_FUSED", "1") != "0"
        # ... on the valid tokens only (pads compacted away); SEQREC_CE_COMPACT=0 keeps the full token axis
        self.ce_compact = os.environ.get("SEQREC_CE_COMPACT", "1") != "0"
        self.ids_wait_early = os.environ.get("SEQREC_IDS_WAIT_EARLY", "1") != "0"
        self.dp_serial = os.environ.get("SEQREC_DP_SERIAL", "0") == "1"   # diagnosis: every collective joined at once
        self.Hk = (self.H + 63) // 64 * 64
        self.Vp = (self.V + 7) // 8 * 8
        self._w_version = 0
        self._split_version = -1
        self.Bt_hi = self.Bt_lo = self.Wb_hi = self.Wb_lo = None
        self.Wt_items = None                      # fp32 W_out^T (V, H) of the candidate scorers, made on first use
        self._wt_version = -1
        if weights is not None:
            self.set_weights(weights)

    # ------------------------------------------------------------------------------------------------ plumbing
    def _mark(self, name):
        """Phase boundary for bench.py's per-kernel timing: a CUDA event on the launching stream."""
        if self.prof is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream(self.device))
            self.prof.append((name, ev))

    def phase_times_ms(self):
        """Elapsed ms between consecutive marks, summed per phase name (call after a synchronize)."""
        out = {}
        for (name, ev), (_, nxt) in zip(self.prof[:-1], self.prof[1:]):
            if name != "end":
                out[name] = out.get(name, 0.0) + ev.elapsed_time(nxt)
        return out

    @property
    def stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @contextlib.contextmanager
    def _branch(self):
        """Work issued inside runs on the side stream, after everything queued on the current stream so far; the caller
        MUST `_join()` before anything consumes its results (and before the step ends).  Serial (a plain pass-through)
        while bench.py profiles phases, so that every phase is timed alone."""
        if not self.overlap or self.prof is not None or self._side_stream is None:
            yield
            return
        self._side_stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self._side_stream):
            yield
        self._branched = True

    def _join(self):
        if getattr(self, "_branched", False):
            torch.cuda.current_stream(self.device).wait_stream(self._side_stream)
            self._branched = False

    def _ce_splits(self, N):
        tiles = (N + 63) // 64
        v_tiles = (self.V + 63) // 64
        s = max(1, min(v_tiles, math.ceil(2 * NUM_SMS / tiles)))
        return s

    def _tc_plan(self, N):
        """Which logits kernels serve a batch of N tokens."""
        big = self.tc_mode != "off" and self.V >= 256 and N >= 128
        fwd = big and self.Hk <= 256
        bwd = fwd
        splits = _lib.load().seqrec_ce_tc_partials(N, 0, self.V) if fwd else 0   # partial rows the TC forward writes
        # hidden sizes above 256 (tune_params_msnbc.py:53 sweeps z_dim up to 1000): the fused kernels keep a [128 x Hk]
        # fp32 accumulator in tensor memory, which ends at Hk = 256 next to the logits tile -- wider layers run the
        # logits path as plain tcgen05 GEMMs over token PANELS (seqrec_gemm_tc, K-looped over any Hk): a panel of logits
        # is materialised, never the (N,V) matrix
        panel = self.Hk > 256 and not self.vocab_parallel
        return dict(fwd=fwd, bwd=bwd, splits=splits, panel=panel, panel_tc=panel and big)

    def _stage_weight_operands(self):
        """bf16 hi/lo copies of W_out (as W and as W^T), refreshed whenever the weights changed."""
        if self._split_version == self._w_version:
            return
        bf = torch.bfloat16
        if self.Bt_hi is None:
            self.Bt_hi = torch.zeros((self.V, self.Hk), dtype=bf, device=self.device)
            self.Wb_hi = torch.zeros((self.Hk, self.Vp), dtype=bf, device=self.device)
            if self.tc_x3:
                self.Bt_lo = torch.zeros((self.V, self.Hk), dtype=bf, device=self.device)
                self.Wb_lo = torch.zeros((self.Hk, self.Vp), dtype=bf, device=self.device)
        st = self.stream
        # W (H, V; ld Vp) and W^T (V, H; ld Hk) from one read of W_out
        call("seqrec_split_bf16_both", ptr(self.W_out), None, ptr(self.Wb_hi), ptr(self.Wb_lo), ptr(self.Bt_hi),
             ptr(self.Bt_lo), self.H, self.V, self.Vp, self.Hk, st)
        self._split_version = self._w_version

    def work(self, B, T):
        key = (B, T)
        w = self._work.get(key)
        if w is None:
            if len(self._work) > 4:
                self._work.clear()
            w = self._work[key] = _Work(self, B, T)
        return w

    def weight_list(self):
        ws = [self.W_in, self.U, self.b, self.W_out]
        if self.out_bias:
            ws.append(self.b_out)
        return ws

    def get_weights(self):
        """Keras `get_weights()` order: [W_in, U, b, W_out (, b_out)] as float32 numpy arrays (full catalog width: the
        column shards of a vocabulary-parallel model are gathered)."""
        out = []
        for i, w in enumerate(self.weight_list()):
            if self.vocab_parallel and i >= 3:
                full = self.comm.all_gather_cat(w.detach().t().contiguous() if w.dim() == 2 else w.detach())
                w = full.t() if w.dim() == 2 else full
            out.append(w.detach().cpu().numpy().copy())
        return out

    def set_weights(self, weights, sync=True):
        """weights: full-catalog arrays in `get_weights()` order (a vocabulary-parallel model keeps its column shard).
        sync: in a multi-process run every rank takes RANK 0's arrays (one broadcast per weight), so replicas can never
        start from different weights -- e.g. when each process drew its own random initialisation."""
        ws = self.weight_list()
        if len(weights) != len(ws):
            raise ValueError("expected %d weight arrays, got %d" % (len(ws), len(weights)))
        for i, (dst, src) in enumerate(zip(ws, weights)):
            src = np.asarray(src, dtype=np.float32)
            full_shape = tuple(dst.shape)
            if self.vocab_parallel and i >= 3:
                full_shape = full_shape[:-1] + (self.V_total,)
            if tuple(src.shape) != full_shape:
                raise ValueError("weight shape %s does not match %s" % (src.shape, full_shape))
            if sync and self.comm.enabled:
                t = torch.from_numpy(np.ascontiguousarray(src)).to(self.device)
                self.comm.broadcast(t, 0)
                if self.vocab_parallel and i >= 3:
                    t = t[..., self.v_lo:self.v_lo + self.V]
                dst.copy_(t)
            else:
                if self.vocab_parallel and i >= 3:
                    src = src[..., self.v_lo:self.v_lo + self.V]
                dst.copy_(torch.from_numpy(np.ascontiguousarray(src)))
        self._w_version += 1

    def get_accumulator(self, name):
        """Adagrad accumulator of one weight (state checkpoints)."""
        return self.get_weight(name, prefix="a")

    def set_accumulator(self, name, value):
        self.set_weight(name, value, prefix="a")

    def get_moments(self, name):
        """Adam's (m, v) of one weight, full width (state checkpoints)."""
        return self.get_weight(name, prefix="m"), self.get_weight(name, prefix="a")

    def set_moments(self, name, m, v):
        self.set_weight(name, m, prefix="m")
        self.set_weight(name, v, prefix="a")

    def get_iterations(self):
        """Optimizer updates applied since set_optimizer (Keras `optimizer.iterations`)."""
        return int(self.iterations.item())

    def set_iterations(self, k):
        self.iterations.fill_(int(k))

    def get_weight(self, name, prefix=""):
        """One weight by name ('W_in', 'U', 'b', 'W_out', 'b_out') as a full-width float32 numpy array."""
        t = getattr(self, prefix + name)
        if self.vocab_parallel and name in ("W_out", "b_out"):
            full = self.comm.all_gather_cat(t.detach().t().contiguous() if t.dim() == 2 else t.detach())
            t = full.t() if t.dim() == 2 else full
        return t.detach().cpu().numpy().copy()

    def set_weight(self, name, value, sync=True, prefix=""):
        t = getattr(self, prefix + name)
        v = np.asarray(value, dtype=np.float32)
        sharded = self.vocab_parallel and name in ("W_out", "b_out")
        full_shape = tuple(t.shape[:-1]) + (self.V_total,) if sharded else tuple(t.shape)
        if tuple(v.shape) != full_shape:
            raise ValueError("weight %s: shape %s does not match %s" % (name, v.shape, full_shape))
        d = torch.from_numpy(np.ascontiguousarray(v)).to(self.device)
        if sync:
            self.comm.broadcast(d, 0)
        t.copy_(d[..., self.v_lo:self.v_lo + self.V] if sharded else d)
        self._w_version += 1

    def reset_optimizer_state(self):
        self.flat_a.zero_()
        self.aW_in.zero_()
        if self.flat_m is not None:
            self.flat_m.zero_()
            self.mW_in.zero_()
        self.iterations.zero_()

    def set_optimizer(self, kind="adagrad", lr=0.01, epsilon=1e-8, clipnorm=0.0, decay=0.0, beta_1=0.9, beta_2=0.999):
        """Adagrad (the reference's optimizer, experiments_methods.py:41) or Keras Adam; resets the optimizer state."""
        self.opt = _optimizer_spec(kind, lr, epsilon, clipnorm, decay, beta_1, beta_2)
        if kind == "adam" and self.flat_m is None:
            self.flat_m = torch.zeros_like(self.flat_a)
            self.mU, self.mb, self.mW_out, self.mb_out = self._views(self.flat_m)
            self.mW_in = torch.zeros_like(self.aW_in)
        self.reset_optimizer_state()

    # ------------------------------------------------------------------------------------------------ batch ingest
    def _zero_step_scalars(self, grads=False):
        """n_valid, n_rows and sumsq start every step at zero; staging a batch is the start of a step.  grads: a
        training step -- the flat gradient buffer (dense, accumulated into by the backward kernels) goes with them."""
        (self._grads_and_scal if grads else self.scal).zero_()

    def _format(self, w, have_t=True, grads=False):
        """(B,T) device ids/targets -> time-major ids/targets/mask + valid-token count (the in-graph part of ingest).
        Ids >= F / targets >= V become pads and raise the device error flag (see check_errors)."""
        self._zero_step_scalars(grads)
        n_in = self.F if w.x_dense is None else 1 << 30
        call("seqrec_format_batch", ptr(w.ids_bt), ptr(w.tgt_bt) if have_t else None, ptr(w.ids),
             ptr(w.tgt) if have_t else None, ptr(w.mask), ptr(w.n_valid_i), w.B, w.T, n_in, self.V_total,
             ptr(self.err_flag), self.stream)

    def check_errors(self):
        """Raise if a staged batch held an item id outside the input table or a target outside the catalog (the
        reference raises IndexError in np_utils.to_categorical, preprocessor.py:75-78).  Host arrays are checked when
        they are staged; device-resident batches are checked by the formatter kernel, which masks the offending token
        and raises a flag -- read here (one 4-byte D2H; called by the model surface once per epoch / call)."""
        bits = int(self.err_flag.item())
        if bits:
            self.err_flag.zero_()
            what = [n for b, n in ((1, "input item id >= %d" % self.F), (2, "target id outside [0, %d)" % self.V_total))
                    if bits & b]
            raise ValueError("batch holds an out-of-range id: " + " and ".join(what))

    def _check_host_ids(self, ids, tgt):
        if ids is not None and not isinstance(ids, torch.Tensor):
            a = np.asarray(ids)
            if a.size and int(a.max()) >= self.F:
                raise ValueError("input item id %d is outside the input table (%d rows)" % (int(a.max()), self.F))
        if tgt is not None and not isinstance(tgt, torch.Tensor):
            a = np.asarray(tgt)
            if a.size and int(a.max()) >= self.V_total:
                raise ValueError("target id %d is outside the catalog (%d items)" % (int(a.max()), self.V_total))

    def _stage(self, w, ids, tgt, x_dense=None, format_now=True, grads=False):
        """Host (numpy / pinned torch) or device batch -> time-major device buffers.  ids (B,T) int32, pad < 0."""
        self._check_host_ids(ids if x_dense is None else None, tgt)

        def to_dev(dst, pin, src):
            if src is None:
                return None
            if isinstance(src, torch.Tensor):
                dst.copy_(src, non_blocking=True)      # device source, or pinned host source: asynchronous either way
            else:
                # the pinned staging buffer is reused every call: wait until the previous asynchronous copy out of it
                # has really run (with CUDA-graph replay the host can be a whole step ahead of the device)
                if w.pin_event is not None:
                    w.pin_event.synchronize()
                pin.copy_(torch.from_numpy(np.ascontiguousarray(src, dtype=np.int32)))
                dst.copy_(pin, non_blocking=True)
                w.pin_dirty = True
            return dst

        w.x_dense = None
        have_t = tgt is not None
        if x_dense is None:
            to_dev(w.ids_bt, w.pin_ids, ids)
        else:
            # dense-feature input (RNNBaseline): x_dense (B,T,F) float; mask = any(x != 0) (model.py:246)
            xd = x_dense if isinstance(x_dense, torch.Tensor) else torch.from_numpy(
                np.ascontiguousarray(x_dense, dtype=np.float32))
            xd = xd.to(self.device, dtype=torch.float32, non_blocking=True)
            w.x_dense = xd.permute(1, 0, 2).contiguous()
            w.ids_bt.copy_(torch.where((xd != 0).any(dim=-1), 0, -1).to(torch.int32))
        if have_t:
            to_dev(w.tgt_bt, w.pin_tgt, tgt)
        if w.pin_dirty:
            w.pin_event = torch.cuda.Event()
            w.pin_event.record(torch.cuda.current_stream(self.device))
            w.pin_dirty = False
        if format_now:
            self._format(w, have_t, grads)

    def _dropout(self, shape, rate):
        t = torch.empty(shape, dtype=torch.float32, device=self.device)
        n = t.numel()
        call("seqrec_dropout_mask_dev", ptr(t), n, float(rate), self.seed, ptr(self.rng_state), self.stream)
        return t

    # ------------------------------------------------------------------------------------------------ forward
    def _forward_hidden(self, w, training, state=None):
        """state: RecurrentState the scan starts from (inference only); None = zeros."""
        st = self.stream
        w.in_scale = None
        w.hscale = None
        w.tc_operands_fresh = False
        self._mark("gather")
        if w.x_dense is None:
            if training and self.dropout_in > 0:
                w.in_scale = self._dropout((w.N,), self.dropout_in)
            call("seqrec_gather_rows", ptr(self.W_in), ptr(self.b), ptr(w.ids), ptr(w.mask), ptr(w.in_scale),
                 ptr(w.xg), w.N, self.F, self.GH, st)
        else:
            if training and self.dropout_in > 0:
                # (RNNBaseline has no input dropout; a y_to_z_dropout model is fed one-hot / id batches, which take the
                #  gather path above -- an element-wise mask over a dense (N, F) input is not built, so say so)
                raise NotImplementedError("y_to_z_dropout on a dense (non one-hot) input batch")
            # K2: time-batched dense input projection (RNNBaseline with [onehot || xs]) -- tcgen05 GEMM when it fills tiles
            gemm(self, w.x_dense.view(w.N, self.F), self.W_in, w.xg.view(w.N, self.GH), "nn", bias=self.b)
        self._mark("rnn_fwd")
        w.rec_mask = None
        if training and self.dropout_rec > 0:
            # one inverted-dropout mask per gate block, (G, B, H), constant over the T steps of this batch; such a step
            # runs on the generic fp32 scan (the tensor-core / register scans share one h operand between the gates)
            w.rec_mask = self._dropout((self.G, w.B, self.H), self.dropout_rec)
            call("seqrec_rnn_forward_rd", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(w.rec_mask),
                 ptr(w.mask), ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
        elif state is not None:
            h0, c0 = self._state_operands(state, w.B)
            if self.rnn_tc:
                call("seqrec_split_bf16", ptr(self.U), None, ptr(self.Ut_hi), ptr(self.Ut_lo), self.H, self.GH, self.H,
                     1, st)
                call("seqrec_rnn_tc_forward_state", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.Ut_hi),
                     ptr(self.Ut_lo), ptr(h0), ptr(c0), ptr(w.mask), ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
            else:
                call("seqrec_rnn_forward_state", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(h0),
                     ptr(c0), ptr(w.mask), ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
        elif self.rnn_tc:
            call("seqrec_split_bf16", ptr(self.U), None, ptr(self.Ut_hi), ptr(self.Ut_lo), self.H, self.GH, self.H, 1,
                 st)
            call("seqrec_rnn_tc_forward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.Ut_hi), ptr(self.Ut_lo),
                 ptr(w.mask), ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
        else:
            call("seqrec_rnn_forward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(w.mask),
                 ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
        self._mark("misc")
        if training and self.dropout_out > 0:
            w.hscale = self._dropout((w.N, self.H), self.dropout_out)

    def _rnn_backward(self, w):
        """K4: dL/dhout (w.dh) -> dxp in place of the saved gates (w.xg)."""
        st = self.stream
        if w.rec_mask is not None:
            call("seqrec_transpose", ptr(self.U), ptr(self.Ut), self.H, self.GH, st)
            call("seqrec_rnn_backward_rd", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.Ut), ptr(w.rec_mask),
                 ptr(w.mask), ptr(w.hout), ptr(w.cst), ptr(w.dh), w.T, w.B, self.H, st)
            return
        if self.rnn_tc:
            call("seqrec_split_bf16", ptr(self.U), None, ptr(self.U_hi), ptr(self.U_lo), self.H, self.GH, self.GH, 0,
                 st)
            call("seqrec_rnn_tc_backward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U_hi), ptr(self.U_lo),
                 ptr(w.mask), ptr(w.hout), ptr(w.cst), ptr(w.dh), w.T, w.B, self.H, st)
            return
        if self._needs_ut:
            call("seqrec_transpose", ptr(self.U), ptr(self.Ut), self.H, self.GH, st)
        call("seqrec_rnn_backward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(self.Ut), ptr(w.mask),
             ptr(w.hout), ptr(w.cst), ptr(w.dh), w.T, w.B, self.H, st)

    def _rnn_weight_grad(self, w):
        """dU, db from dxp (w.xg), hout and (GRU) r*h_{t-1} (w.cst)."""
        st = self.stream
        if w.rec_mask is not None:
            if w.rd_scratch is None:
                w.rd_scratch = torch.empty((w.T, w.B, self.H), dtype=torch.float32, device=self.device)
            call("seqrec_rnn_weight_grad_rd", CELL[self.cell], ptr(w.xg), ptr(w.hout), ptr(w.cst), ptr(w.rec_mask),
                 ptr(w.rd_scratch), ptr(self.dU), ptr(self.db), w.T, w.B, self.H, st)
            return
        if self.wgrad_tc:
            if w.D_hi is None:
                bf = torch.bfloat16
                w.D_hi = torch.empty((w.N, self.GH), dtype=bf, device=self.device)
                w.D_lo = torch.empty((w.N, self.GH), dtype=bf, device=self.device)
                w.Hs_hi = torch.empty((w.N, self.H), dtype=bf, device=self.device)
                w.Hs_lo = torch.empty((w.N, self.H), dtype=bf, device=self.device)
                if self.cell == "GRU":
                    w.C_hi = torch.empty((w.N, self.H), dtype=bf, device=self.device)
                    w.C_lo = torch.empty((w.N, self.H), dtype=bf, device=self.device)
            # dxp -> bf16 hi/lo and db = column sums, one pass (rows chunked over blockIdx.y: 65535 * 32 rows at most)
            fused_db = w.N <= 65535 * 32
            if fused_db:
                call("seqrec_split_bf16_colsum", ptr(w.xg), ptr(w.D_hi), ptr(w.D_lo), ptr(self.db), w.N, self.GH, st)
            else:
                call("seqrec_split_bf16", ptr(w.xg), None, ptr(w.D_hi), ptr(w.D_lo), w.N, self.GH, self.GH, 0, st)
            hs_hi, hs_lo = w.Hs_hi, w.Hs_lo
            if w.tc["fwd"] and self.tc_x3 and w.hscale is None and self.Hk == self.H and w.tc_operands_fresh:
                hs_hi, hs_lo = w.A_hi, w.A_lo              # the logits kernels' operand IS bf16 hi/lo of hout
            else:
                call("seqrec_split_bf16", ptr(w.hout), None, ptr(w.Hs_hi), ptr(w.Hs_lo), w.N, self.H, self.H, 0, st)
            if self.cell == "GRU":
                call("seqrec_split_bf16", ptr(w.cst), None, ptr(w.C_hi), ptr(w.C_lo), w.N, self.H, self.H, 0, st)
            call("seqrec_rnn_weight_grad_tc", CELL[self.cell], ptr(w.xg), ptr(w.D_hi), ptr(w.D_lo), ptr(hs_hi),
                 ptr(hs_lo), ptr(w.C_hi), ptr(w.C_lo), ptr(self.dU), None if fused_db else ptr(self.db), w.T, w.B,
                 self.H, st)
            return
        call("seqrec_rnn_weight_grad", CELL[self.cell], ptr(w.xg), ptr(w.hout), ptr(w.cst), ptr(self.dU), ptr(self.db),
             w.T, w.B, self.H, st)

    def _forward_ce(self, w, with_targets=True, training=False, train=False):
        if w.tc["panel"]:
            return self._ce_panels(w, with_targets, train=train, backward=False)
        n_splits = self._ce_partials(w, with_targets, training)
        self._finalize_ce(w, w.ws_m, w.ws_s, n_splits, with_targets, train)

    def _ce_partials(self, w, with_targets=True, training=False):
        """Logits kernels only: per-token partial (max, sum-exp) rows in w.ws_m / w.ws_s and the target logit in w.zy.
        Returns the number of partial rows."""
        st = self.stream
        if w.tc["fwd"]:
            self._mark("stage_operands")
            self._stage_weight_operands()
            if training and w.tc["bwd"]:
                call("seqrec_split_bf16_both", ptr(w.hout), ptr(w.hscale), ptr(w.A_hi), ptr(w.A_lo), ptr(w.Ht_hi),
                     ptr(w.Ht_lo), w.N, self.H, self.Hk, w.Np, st)
            else:
                call("seqrec_split_bf16", ptr(w.hout), ptr(w.hscale), ptr(w.A_hi), ptr(w.A_lo), w.N, self.H, self.Hk,
                     0, st)
            w.tc_operands_fresh = True
            self._join()                          # W_out operands staged on the branch by _train_core
            self._mark("ce_fwd")
            if with_targets:                      # the target logit is not needed before the finalize kernel
                with self._branch():
                    call("seqrec_target_logit", ptr(w.hout), ptr(w.hscale), ptr(self.W_out), ptr(self.b_out),
                         ptr(w.tgt), ptr(w.zy), w.N, self.H, self.V, None, None, self.stream)
            call("seqrec_ce_tc_forward", ptr(w.A_hi), ptr(w.A_lo), ptr(self.Bt_hi), ptr(self.Bt_lo), ptr(self.b_out),
                 ptr(w.ws_m), ptr(w.ws_s), w.N, self.Hk, self.V, 0, self.V, 1 if self.tc_x3 else 0, st)
            self._join()
            n_splits = w.tc["splits"]
        else:
            self._mark("ce_fwd")
            n_splits = self._ce_splits(w.N)
            call("seqrec_ce_forward", ptr(w.hout), ptr(w.hscale), ptr(self.W_out), ptr(self.b_out),
                 ptr(w.tgt) if with_targets else None, ptr(w.ws_m), ptr(w.ws_s), ptr(w.zy), w.N, self.H, self.V, 0,
                 self.V, self.V, n_splits, st)
        return n_splits

    def _finalize_ce(self, w, ws_m, ws_s, n_splits, with_targets=True, train=False):
        """train: a training step -- the loss sum and the unmasked-token count go (as floats) into the step-float block
        at the head of the gradient buffer (reduced over ranks together with dU / db), and the local masked-mean loss
        into w.loss_mean."""
        if train:
            call("seqrec_ce_finalize_mean", ptr(ws_m), ptr(ws_s), ptr(w.zy), ptr(w.mask), ptr(w.m), ptr(w.s), ptr(w.ce),
                 ptr(w.py), ptr(w.coef), ptr(self.step_loss_sum), ptr(w.n_valid_i), ptr(self.n_valid_f),
                 ptr(w.loss_mean), w.N, n_splits, None, self.stream)
        else:
            call("seqrec_ce_finalize", ptr(ws_m), ptr(ws_s), ptr(w.zy) if with_targets else None, ptr(w.mask),
                 ptr(w.m), ptr(w.s), ptr(w.ce), ptr(w.py), ptr(w.coef), ptr(w.loss_sum), w.N, n_splits, self.stream)
        self._mark("misc")

    def _ce_panels(self, w, with_targets=True, train=False, backward=False):
        """Logits path for hidden sizes above 256, on the tcgen05 GEMM (csrc/gemm_tc.cu, K-looped): the tokens are walked
        in PANELS of `nb` rows; per panel  Z = hs . W_out (+ b_out)  is materialised (nb x V fp32, <= 256 MB), reduced to
        the per-token softmax statistics, turned into dlogit in place and consumed by  dh = dZ . W_out^T  and
        dW_out += hs^T . dZ  -- three logits-sized GEMMs per step, none recomputed.  The full (N,V) matrix never exists."""
        st = self.stream
        N, H, Hk, V = w.N, self.H, self.Hk, self.V
        x3 = 1 if self.tc_x3 else 0
        tc = w.tc["panel_tc"]                     # False: shapes that do not fill tensor-core tiles (e.g. the 17-item
        hs_all = None                             # MSNBC catalog), or tc='off': the same panels on the fp32 SIMT GEMMs
        if tc:
            self._mark("stage_operands")
            self._stage_weight_operands()
            call("seqrec_split_bf16_both", ptr(w.hout), ptr(w.hscale), ptr(w.A_hi), ptr(w.A_lo), ptr(w.Ht_hi),
                 ptr(w.Ht_lo), N, H, Hk, w.Np, st)
        else:
            hs_all = w.hout.view(N, H) if w.hscale is None else w.hout.view(N, H) * w.hscale.view(N, H)
        w.tc_operands_fresh = False
        self._join()
        self._mark("ce_fwd")
        if with_targets:
            call("seqrec_target_logit", ptr(w.hout), ptr(w.hscale), ptr(self.W_out), ptr(self.b_out), ptr(w.tgt),
                 ptr(w.zy), N, H, V, None, None, st)
        nb_max = max(128, min((N + 127) // 128 * 128, ((256 << 20) // (4 * V)) // 128 * 128))
        if w.pz is None or w.pz.shape[0] < nb_max:
            bf = torch.bfloat16
            Vk, nbk = (V + 63) // 64 * 64, nb_max
            w.pz = torch.empty((nb_max, V), dtype=torch.float32, device=self.device)
            if tc:
                w.pz_hi = torch.zeros((nb_max, Vk), dtype=bf, device=self.device)
                w.pz_lo = torch.zeros((nb_max, Vk), dtype=bf, device=self.device) if x3 else None
                w.pzt_hi = torch.zeros((V, nbk), dtype=bf, device=self.device)
                w.pzt_lo = torch.zeros((V, nbk), dtype=bf, device=self.device) if x3 else None
        if tc:
            Vk, nbk = w.pz_hi.shape[1], w.pzt_hi.shape[1]
        n_panels = (N + nb_max - 1) // nb_max
        parts = torch.zeros(n_panels, dtype=torch.float32, device=self.device)
        el = 2                                                       # bytes per bf16
        for p, n0 in enumerate(range(0, N, nb_max)):
            nb = min(nb_max, N - n0)
            off = lambda t, elems, size: ctypes.c_void_p(t.data_ptr() + elems * size) if t is not None else None
            sl = slice(n0, n0 + nb)
            Z = w.pz[:nb]
            if tc:
                call("seqrec_gemm_tc", off(w.A_hi, n0 * Hk, el), off(w.A_lo, n0 * Hk, el), ptr(self.Bt_hi),
                     ptr(self.Bt_lo), ptr(self.b_out), ptr(Z), nb, V, Hk, Hk, Hk, V, 0, x3, st)
            else:
                call("seqrec_gemm_nn", ptr(hs_all[sl]), ptr(self.W_out), ptr(self.b_out), ptr(Z), nb, V, H, 0, st)
            m, s_, zy, mask = w.m[sl], w.s[sl], w.zy[sl], w.mask.view(-1)[sl]
            tg = w.tgt.view(-1)[sl]
            call("seqrec_softmax_rows_stats", ptr(Z), None, ptr(m), ptr(s_), None, nb, V, st)
            call("seqrec_ce_finalize", ptr(m), ptr(s_), ptr(zy) if with_targets else None, ptr(mask), ptr(m), ptr(s_),
                 ptr(w.ce[sl]), ptr(w.py[sl]), ptr(w.coef[sl]), ptr(parts[p:p + 1]), nb, 1, st)
            if not backward:
                continue
            call("seqrec_softmax_rows_dlogit", ptr(Z), ptr(tg), ptr(m), ptr(s_), ptr(w.coef[sl]), nb, V, st)
            if self.db_out is not None:
                call("seqrec_colsum", ptr(Z), ptr(self.db_out), nb, V, V, st)
            dh = w.dh.view(N, H)[sl]
            if tc:
                call("seqrec_split_bf16_both", ptr(Z), None, ptr(w.pz_hi), ptr(w.pz_lo), ptr(w.pzt_hi), ptr(w.pzt_lo), nb,
                     V, Vk, nbk, st)
                # dh[panel] = dZ . W_out^T   (K = V; W_out rows are K-major over the items: the Wb operand)
                call("seqrec_gemm_tc", ptr(w.pz_hi), ptr(w.pz_lo), ptr(self.Wb_hi), ptr(self.Wb_lo), None, ptr(dh), nb, H,
                     V, Vk, self.Vp, H, 0, x3, st)
                # dW_out += hs[panel]^T . dZ   (K = the panel's tokens: Ht columns [n0, n0 + nb), dZ^T rows)
                call("seqrec_gemm_tc", off(w.Ht_hi, n0, el), off(w.Ht_lo, n0, el), ptr(w.pzt_hi), ptr(w.pzt_lo), None,
                     ptr(self.dW_out), H, V, nb, w.Np, nbk, V, 1, x3, st)
            else:
                call("seqrec_gemm_nt", ptr(Z), ptr(self.W_out), ptr(dh), nb, H, V, V, V, H, 0, st)
                call("seqrec_gemm_tn_atomic", ptr(hs_all[sl]), ptr(Z), ptr(self.dW_out), H, V, nb, st)
            if w.hscale is not None:
                dh.mul_(w.hscale.view(N, H)[sl])
        if train:
            torch.sum(parts, dim=0, keepdim=True, out=self.step_loss_sum)
            self.n_valid_f.copy_(w.n_valid_i)
            torch.div(self.step_loss_sum, self.n_valid_f, out=w.loss_mean)
        else:
            torch.sum(parts, dim=0, keepdim=True, out=w.loss_sum)
        self._mark("misc")

    def _ce_train_fused(self, w, zy_reduce=None, s_reduce=None):
        """Training-step logits pass on the tensor cores, fused: statistics + dh from ONE logits computation
        (seqrec_ce_tc_fused), finalize, dh finish.  Leaves w.m (= the per-token reference logit), w.s, w.coef ready for
        the item-stationary dW kernel.  zy_reduce / s_reduce: vocabulary-parallel hooks that sum the target logit and
        the partial sum-exp over the item shards.

        The token axis is COMPACTED first (self.ce_compact): pad tokens carry neither loss nor gradient, so operands and
        per-token arrays hold the valid tokens only (ascending time-major order) and every logits-sized GEMM of the step
        shrinks by the padding fraction; dh is scattered back to the full [T][B][H] layout by the finish kernel.  The
        valid count lives on the device (w.n_c): a captured step replays with any amount of padding."""
        st = self.stream
        cp = self.ce_compact
        self._mark("stage_operands")
        self._stage_weight_operands()
        if cp:
            if w.orig is None:
                i32 = torch.int32
                w.orig = torch.zeros(w.N, dtype=i32, device=self.device)
                w.tgt_c = torch.zeros(w.N, dtype=i32, device=self.device)
                w.n_c = torch.zeros(1, dtype=i32, device=self.device)
                w.blk = torch.zeros((w.N + 255) // 256, dtype=i32, device=self.device)
                w.acc = torch.empty((w.N, self.H), dtype=torch.float32, device=self.device)
            call("seqrec_compact_tokens", ptr(w.mask), ptr(w.tgt), w.N, ptr(w.orig), ptr(w.tgt_c), ptr(w.n_c),
                 ptr(w.blk), st)
            call("seqrec_split_bf16_both_rows", ptr(w.hout), ptr(w.hscale), ptr(w.orig), ptr(w.n_c), ptr(w.A_hi),
                 ptr(w.A_lo), ptr(w.Ht_hi), ptr(w.Ht_lo), w.N, self.H, self.Hk, w.Np, st)
            w.tc_operands_fresh = False           # A holds compacted rows: not the dU GEMM's hout operand
            tgt, mask, orig, n_c, acc = w.tgt_c, None, w.orig, w.n_c, w.acc
        else:
            call("seqrec_split_bf16_both", ptr(w.hout), ptr(w.hscale), ptr(w.A_hi), ptr(w.A_lo), ptr(w.Ht_hi),
                 ptr(w.Ht_lo), w.N, self.H, self.Hk, w.Np, st)
            w.tc_operands_fresh = True
            tgt, mask, orig, n_c, acc = w.tgt, w.mask, None, None, w.dh
        w.ce_tgt, w.ce_n = tgt, n_c               # what the dW kernel indexes with
        self._join()                              # W_out operands staged on the branch by the caller
        self._mark("ce_fwd")
        call("seqrec_target_logit", ptr(w.hout), ptr(w.hscale), ptr(self.W_out), ptr(self.b_out), ptr(tgt),
             ptr(w.zy), w.N, self.H, self.V, ptr(orig), ptr(n_c), st)
        if zy_reduce is not None:
            zy_reduce(w.zy)
        self._mark("ce_fwd:zero")
        w.dh.zero_()
        if cp:
            acc.zero_()
        w.s.zero_()
        self._mark("ce_fwd:fused")
        call("seqrec_ce_tc_fused", ptr(w.A_hi), ptr(w.A_lo), ptr(self.Bt_hi), ptr(self.Bt_lo), ptr(self.Wb_hi),
             ptr(self.Wb_lo), ptr(w.zy), ptr(mask), ptr(self.b_out), ptr(acc), ptr(w.s), w.N, self.H, self.Hk,
             self.V, self.Vp, 0, self.V, 1 if self.tc_x3 else 0, ptr(n_c), st)
        self._mark("ce_fwd:finalize")
        if s_reduce is not None:
            s_reduce(w.s)
        call("seqrec_ce_finalize_mean", ptr(w.zy), ptr(w.s), ptr(w.zy), ptr(mask), ptr(w.m), ptr(w.s), ptr(w.ce),
             ptr(w.py), ptr(w.coef), ptr(self.step_loss_sum), ptr(w.n_valid_i), ptr(self.n_valid_f), ptr(w.loss_mean),
             w.N, 1, ptr(n_c), st)
        self._mark("misc")
        call("seqrec_ce_dh_finish", ptr(acc), ptr(w.dh), ptr(w.s), ptr(w.coef), ptr(tgt), ptr(self.Bt_hi),
             ptr(self.Bt_lo), ptr(w.hscale), w.N, self.H, self.Hk, ptr(orig), ptr(n_c), st)

    def _backward_ce(self, w, dh=True):
        """K6.  Gradients leave UN-normalised (dlogit = (p - onehot) * coef, no 1/n_valid): everything downstream is
        linear in that factor, so the optimiser kernels apply 1/n_valid_global once -- which is what lets a
        data-parallel step run its backward pass before the token counts of the other ranks are known.
        dh=False: after the fused pass -- only the item-stationary dW kernel runs, on the (compacted) token axis the
        fused pass left behind."""
        st = self.stream
        if w.tc["bwd"]:
            tgt, n_c = (w.tgt, None) if dh else (w.ce_tgt, w.ce_n)
            call("seqrec_ce_tc_backward", ptr(w.A_hi), ptr(w.A_lo), ptr(w.Ht_hi), ptr(w.Ht_lo), ptr(self.Bt_hi),
                 ptr(self.Bt_lo), ptr(self.Wb_hi), ptr(self.Wb_lo), ptr(tgt), ptr(w.m), ptr(w.s), ptr(w.coef),
                 None, ptr(w.hscale), ptr(w.dh) if dh else None, ptr(self.dW_out), w.N, self.H, self.Hk, self.V,
                 self.Vp, w.Np, 0, self.V, self.V, 0, 1 if self.tc_x3 else 0, ptr(self.b_out), ptr(self.db_out),
                 ptr(n_c), st)
        else:
            call("seqrec_ce_backward", ptr(w.hout), ptr(w.hscale), ptr(self.W_out), ptr(self.b_out), ptr(w.tgt),
                 ptr(w.m), ptr(w.s), ptr(w.coef), None, ptr(w.dh), ptr(self.dW_out), ptr(self.db_out),
                 w.N, self.H, self.V, 0, self.V, self.V, 0, st)

    # ------------------------------------------------------------------------------------------------ public steps
    def loss_batch(self, ids, tgt, x_dense=None):
        """Forward only: returns (loss_sum, n_valid) device tensors of THIS rank's batch (evaluate path)."""
        w = self._scan_batch(ids, tgt, x_dense)
        if self.vocab_parallel:
            # loss_sum already covers every rank's tokens: report this rank's share so callers can all-reduce as usual
            wg = self._vp_forward(w, training=False)
            return self._my_rows(wg.ce).sum().reshape(1), w.n_valid_i.to(torch.float32)
        self._forward_ce(w)
        return w.loss_sum.clone(), w.n_valid_i.to(torch.float32)

    def train_batch(self, ids, tgt, x_dense=None):
        """One optimisation step on the global batch (this rank's shard).  Returns the global masked-mean loss as a
        one-element device tensor (no host sync)."""
        if self.opt is None:
            raise _lib.SeqrecError("compile_model / set_optimizer must be called before training")
        B, T = (ids.shape if ids is not None else x_dense.shape[:2])
        w = self.work(int(B), int(T))
        core = self._train_core_vp if self.vocab_parallel else self._train_core
        self._mark("ingest")
        graphable = (self.use_graphs and x_dense is None and self.prof is None and
                     (not self.comm.enabled or self.graph_collectives))
        if not graphable:
            self._stage(w, ids, tgt, x_dense, grads=True)
            return core(w)
        # CUDA-graph replay of the whole step (fixed shapes and buffers): the ~22 launches of a step -- and the NCCL
        # calls of a multi-GPU step -- are submitted as one graph, which removes the launch gaps between them.  The
        # first step of a (B,T) shape runs eagerly, the second one captures.
        self._stage(w, ids, tgt, None, format_now=False)
        key = self._graph_key()
        if w.graph is not None and w.graph_key != key:
            w.graph, w.graph_calls = None, 1      # host state baked into the captured launches changed: re-capture
        if w.graph is None:
            w.graph_calls += 1
            if w.graph_calls < 2:
                self._format(w, grads=True)
                return core(w)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            # no garbage collection inside the capture: collecting an unreachable work object frees its pinned staging
            # buffers, and the host allocator's event queries then invalidate the capture
            gc_was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(g):
                    self._format(w, grads=True)
                    w.graph_loss = core(w)
            finally:
                if gc_was_on:
                    gc.enable()
            w.graph, w.graph_key = g, key
        w.graph.replay()
        self._w_version += 1
        return w.graph_loss

    def _graph_key(self):
        """Everything a captured step bakes in BY VALUE (kernel arguments and which kernels are launched at all)."""
        o = self.opt
        return (o["lr"], o["eps"], o["clipnorm"], tuple(sorted(self.trainable.items())), self.dropout_in,
                self.dropout_out, self.dropout_rec, self.overlap, self.ce_fused, self.ce_compact, self.rnn_tc, self.wgrad_tc, self.tc_mode, self.tc_x3,
                o["kind"], o["beta_1"], o["beta_2"], o["decay"])

    def _train_core(self, w):
        """forward + backward + exchange + update on the staged batch (everything after the host->device copy).

        Data parallel (SURVEY 8(e)): no collective sits between the forward and the backward pass.  The backward runs
        un-normalised; [n_valid, loss_sum] ride in the step-float block that sits between dW_in and dU | db in ONE
        gradient allocation and are summed over the ranks together with a neighbour: with dW_in (dense exchange of a
        small catalog; started right after the scatter-add, it travels behind the dU GEMMs) or with dU | db.  dW_out /
        db_out are reduced behind the recurrent backward pass.  The optimiser kernels then divide by the global
        n_valid.  Three all-reduces per step (two in the row-exchange mode), none of them blocking a kernel launch."""
        st = self.stream
        comm = self.comm
        self._split_version = -1                  # a training step always follows a weight update: re-stage W_out
        dense_rows = (comm.enabled and w.x_dense is None and
                      embedding_grad_mode(self.F, self.GH, w.N * comm.world) == "dense")
        # union of touched rows for the dense dW_in exchange: the ids of all ranks travel behind the forward pass
        all_ids, ids_handle = comm.all_gather_cat_async(w.ids.view(-1)) if dense_rows else (None, None)
        if ids_handle is not None and self.dp_serial:
            ids_handle.wait()
            ids_handle = None
        if w.tc["fwd"]:
            self._mark("stage_operands")
            with self._branch():                  # bf16 operands of the updated W_out, behind gather + scan
                self._stage_weight_operands()
        self._forward_hidden(w, training=True)
        if ids_handle is not None and self.ids_wait_early:
            # The logits kernels are persistent (one CTA per SM, all of its shared memory): a collective kernel that is
            # still resident on a few SMs -- waiting for a slower rank -- keeps their last CTAs out and doubles their
            # time.  So the ids exchange is joined HERE, behind gather + scan and before the logits kernels start.
            ids_handle.wait()
            ids_handle = None
        fused = self.ce_fused and w.tc["bwd"]
        if w.tc["panel"]:
            self._ce_panels(w, True, train=True, backward=True)      # statistics, dh and dW_out panel by panel
        elif fused:
            self._ce_train_fused(w)
        else:
            self._forward_ce(w, training=True, train=True)

        # ---- backward (the gradient buffer was cleared with the step scalars when the batch was staged)
        self._mark("ce_bwd")
        if not w.tc["panel"]:
            self._backward_ce(w, dh=not fused)
        # dW_out / db_out are final here: their all-reduce runs on NCCL's stream behind the recurrent backward pass
        (o_u, s_u), (o_b, s_b) = self._seg[0], self._seg[1]
        head = o_b + s_b
        pending = [comm.all_reduce_sum(self.flat_g[head:], async_op=True)] if comm.enabled else []
        if self.dp_serial and pending:
            pending.pop().wait()
        self._mark("rnn_bwd")
        self._rnn_backward(w)
        # ---- input-kernel gradient and recurrent weight-gradient GEMMs as parallel branches (both only read dxp)
        branch_wgrad = self.overlap and self.prof is None
        if branch_wgrad:
            with self._branch():
                self._rnn_weight_grad(w)
        self._mark("scatter")
        dense_in = False
        if w.x_dense is None:                     # (n_rows and sumsq were cleared when the batch was staged)
            if not comm.enabled or dense_rows:
                call("seqrec_scatter_add_rows", ptr(w.xg), ptr(w.ids), ptr(w.mask), ptr(w.in_scale), ptr(self.dW_in),
                     ptr(self.touched), ptr(self.rows), ptr(self.n_rows), w.N, self.F, self.GH, st)
                if dense_rows:
                    dense_in = True
                    if ids_handle is not None:
                        ids_handle.wait()
                    call("seqrec_mark_rows", ptr(all_ids), None, ptr(self.touched), ptr(self.rows), ptr(self.n_rows),
                         all_ids.numel(), self.F, st)
            else:
                self._scatter_gathered_rows(w)
        else:
            self.dW_in.zero_()
            gemm(self, w.x_dense.view(w.N, self.F), w.xg.view(w.N, self.GH), self.dW_in, "tn")
            dense_in = comm.enabled
        if comm.enabled and dense_in:
            # dense dW_in (small catalogs) and the step floats [n_valid, loss_sum] are adjacent in the gradient buffer:
            # ONE all-reduce, started as soon as the scatter-add is done -- it travels while the dU GEMMs still run
            pending.append(comm.all_reduce_sum(self._gbuf[:self._fgh + 64], async_op=True))
            if self.dp_serial:
                pending.pop().wait()
        self._mark("rnn_wgrad")
        if branch_wgrad:
            self._join()
        else:
            self._rnn_weight_grad(w)
        self._mark("allreduce")
        if comm.enabled:
            # dU | db (and the step floats in front of them when they did not travel with dW_in)
            lo = self._fgh + 64 if dense_in else self._fgh
            pending.append(comm.all_reduce_sum(self._gbuf[lo:self._fgh + 64 + head], async_op=True))

        # ---- global-norm clip + Adagrad (needs every reduced gradient: clipnorm is global, SURVEY D7)
        for h in pending:
            if h is not None:
                h.wait()
        self._mark("optim")
        self._apply_update(w, scalars_clean=True)
        self._w_version += 1
        if comm.enabled:
            loss = self.step_loss_sum / self.n_valid_f
        else:
            # written by the finalize kernel; a graph replay hands out the static buffer, an eager step a private copy
            loss = w.loss_mean if torch.cuda.is_current_stream_capturing() else w.loss_mean.clone()
        self._mark("end")
        return loss

    def _scatter_gathered_rows(self, w):
        """Row exchange of dW_in (large catalogs): all-gather (ids, dxp rows [, y->z dropout factors]) and scatter-add
        them locally, so every replica applies the identical row-sparse update.  Pads carry id -1 (formatter)."""
        comm = self.comm
        all_ids = comm.all_gather_cat(w.ids.view(-1))
        all_dxp = comm.all_gather_cat(w.xg.view(w.N, self.GH))
        all_scale = comm.all_gather_cat(w.in_scale) if w.in_scale is not None else None
        all_mask = (all_ids >= 0).to(torch.uint8)
        call("seqrec_scatter_add_rows", ptr(all_dxp), ptr(all_ids), ptr(all_mask), ptr(all_scale), ptr(self.dW_in),
             ptr(self.touched), ptr(self.rows), ptr(self.n_rows), all_ids.numel(), self.F, self.GH, self.stream)

    # ------------------------------------------------------------------------------------------------ vocabulary parallel
    def _vp_forward(self, w, training, train=False):
        """Shared by training and evaluation: every rank scores ALL ranks' tokens against its item shard, then the
        per-token (max, sum-exp) partials and the target logit are merged across ranks.  Returns the work object that
        holds the global-token buffers (token order: rank-major blocks of each rank's time-major tokens).
        Three collectives: hidden rows, targets (pads are -1, so the mask travels with them), packed (m, s, zy)."""
        wg, _ = self._vp_gather(w)
        if train:
            # n_valid and the loss sum of ALL tokens are known locally (identical on every rank): they go into the step
            # floats directly and stay outside the reduced range
            self.scal[0:1].copy_(wg.mask.view(-1).sum().to(torch.int32))
        if train and self.ce_fused and wg.tc["bwd"]:
            # fused statistics + dh pass: the target logit (owner's shard) is summed over the shards FIRST and is every
            # rank's reference; the partial sum-exps then add up across shards (same reference) -- two N-float all-reduces
            self._ce_train_fused(wg, zy_reduce=self.comm.all_reduce_sum, s_reduce=self.comm.all_reduce_sum)
            wg.fused = True
            return wg
        wg.fused = False
        self._vp_merge(wg, True, training, train)
        return wg

    def _vp_gather(self, w, last_step_only=False, with_targets=True):
        """All ranks' rows of w -- every token, or step T-1 of every session -- in this rank's work(B*P, T or 1), rank
        after rank: the hidden rows (times the output-dropout factors when set) and either the targets (remapped to
        this shard's item ids, -1 elsewhere; mask = target >= 0) or the mask.  Returns (wg, the gathered global target
        ids or None)."""
        comm = self.comm
        wg = self.work(w.B * comm.world, 1 if last_step_only else w.T)
        rows = w.hout[w.T - 1] if last_step_only else w.hout.view(w.N, self.H)
        if w.hscale is not None:              # output dropout of a training step (every step)
            rows = rows * w.hscale
        wg.hout.view(wg.N, self.H).copy_(comm.all_gather_cat(rows))
        wg.hscale = None
        if not with_targets:
            wg.mask.view(-1).copy_(comm.all_gather_cat(w.mask[w.T - 1] if last_step_only else w.mask.view(-1)))
            return wg, None
        tgt_all = comm.all_gather_cat(w.tgt[w.T - 1] if last_step_only else w.tgt.view(-1))
        wg.mask.view(-1).copy_(tgt_all >= 0)
        local = (tgt_all >= self.v_lo) & (tgt_all < self.v_lo + self.V)
        wg.tgt.view(-1).copy_(torch.where(local, tgt_all - self.v_lo, torch.full_like(tgt_all, -1)))
        wg.zy.zero_()
        return wg, tgt_all

    def _vp_merge(self, wg, with_targets, training=False, train=False):
        """Catalog-wide softmax statistics of wg's rows from this shard's logits: the partials are merged locally to
        (m_r, s_r) per row, ONE exchange of the packed (m, s[, zy]), then the global merge (only the owner of a target
        contributes a non-zero zy)."""
        comm = self.comm
        n_splits = self._ce_partials(wg, with_targets, training)
        call("seqrec_ce_finalize", ptr(wg.ws_m), ptr(wg.ws_s), None, None, ptr(wg.m), ptr(wg.s), None, None, None, None,
             wg.N, n_splits, self.stream)
        parts = [wg.m, wg.s, wg.zy] if with_targets else [wg.m, wg.s]
        packed = comm.all_gather_cat(torch.stack(parts).unsqueeze(0)).permute(1, 0, 2).contiguous()   # (2|3, P, N)
        if with_targets:
            torch.sum(packed[2], dim=0, out=wg.zy)
        self._finalize_ce(wg, packed[0], packed[1], comm.world, with_targets, train=train)

    def _my_rows(self, t):
        """This rank's block of a tensor over all ranks' rows (rank-major blocks)."""
        n = t.shape[0] // self.comm.world
        return t[self.comm.rank * n:(self.comm.rank + 1) * n]

    def _train_core_vp(self, w):
        """Vocabulary-parallel step (SURVEY 8(e), cfg4): data-parallel scan, logits against the local V/P items for the
        tokens of ALL ranks.  Seven collectives per step, all inside the captured graph: all-gather hidden rows / targets
        / packed softmax partials, reduce-scatter dh, ONE all-reduce of [sharded squared norm | dU | db], all-gather ids
        and dxp rows for the row-sparse dW_in."""
        st = self.stream
        comm = self.comm
        self._split_version = -1
        self._forward_hidden(w, training=True)
        wg = self._vp_forward(w, training=True, train=True)
        # ---- backward: dW_out / db_out of the shard are complete locally; dh is summed over the item shards
        self._mark("ce_bwd")
        self._backward_ce(wg, dh=not wg.fused)
        self._mark("allreduce")
        comm.reduce_scatter_sum(w.dh.view(w.N, self.H), wg.dh.view(wg.N, self.H))
        if w.hscale is not None:
            w.dh.view(w.N, self.H).mul_(w.hscale)
        (o_u, s_u), (o_b, s_b) = self._seg[0], self._seg[1]
        head = o_b + s_b
        o = self.opt
        if o["clipnorm"] > 0:
            # squared norm of the SHARDED gradients (summed over ranks below, in the slot right in front of dU);
            # replicated gradients count once
            call("seqrec_sumsq", ptr(self.flat_g[head:]), self.flat_g.numel() - head, ptr(self.sumsq), st)
            self.stepf[63:64].copy_(self.sumsq)
            self.sumsq.zero_()
        self._mark("rnn_bwd")
        self._rnn_backward(w)
        self._mark("rnn_wgrad")
        self._rnn_weight_grad(w)
        self._mark("scatter")
        comm.all_reduce_sum(self._gbuf[self._fgh + 63:self._fgh + 64 + head])
        self._scatter_gathered_rows(w)
        # ---- global norm + update
        max_rows = min(self.F, w.N * comm.world)
        self._mark("optim")
        if o["clipnorm"] > 0:
            self.sumsq.copy_(self.stepf[63:64])
            call("seqrec_sumsq", ptr(self.flat_g[:head]), head, ptr(self.sumsq), st)
            call("seqrec_sumsq_rows", ptr(self.dW_in), ptr(self.rows), ptr(self.n_rows), self.GH, max_rows,
                 ptr(self.sumsq), st)
        if o["kind"] == "adam":
            self._adam(self.flat_p, self.flat_g, self.flat_m, self.flat_a, st)
            self._adam_table(st)
            self.iterations.add_(1)
        else:
            call("seqrec_adagrad", ptr(self.flat_p), ptr(self.flat_g), ptr(self.flat_a), self.flat_p.numel(), o["lr"],
                 o["eps"], o["clipnorm"], ptr(self.sumsq), ptr(self.n_valid_f), st)
            call("seqrec_adagrad_rows", ptr(self.W_in), ptr(self.dW_in), ptr(self.aW_in), ptr(self.rows),
                 ptr(self.n_rows), ptr(self.touched), self.GH, max_rows, o["lr"], o["eps"], o["clipnorm"],
                 ptr(self.sumsq), ptr(self.n_valid_f), st)
        self._w_version += 1
        loss = wg.loss_mean if torch.cuda.is_current_stream_capturing() else wg.loss_mean.clone()
        self._mark("end")
        return loss

    def _segments(self):
        names = ["U", "b", "W_out", "b_out"]
        return [(n, o, s) for n, (o, s) in zip(names, self._seg) if s > 0]

    def _apply_update(self, w, scalars_clean=False):
        st = self.stream
        o = self.opt
        den = ptr(self.n_valid_f)                 # gradients are stored un-normalised: the kernels divide
        if not scalars_clean:
            self.sumsq.zero_()
        segs = self._segments()
        all_dense = all(self.trainable[n] for n, _, _ in segs)
        max_rows = min(self.F, w.N * self.comm.world)
        # the W_in half (row-sparse or dense) runs as a parallel branch of the flat-buffer half
        if o["clipnorm"] > 0:
            if self.trainable["W_in"]:
                with self._branch():
                    if w.x_dense is None:
                        call("seqrec_sumsq_rows", ptr(self.dW_in), ptr(self.rows), ptr(self.n_rows), self.GH, max_rows,
                             ptr(self.sumsq), self.stream)
                    else:
                        call("seqrec_sumsq", ptr(self.dW_in), self.dW_in.numel(), ptr(self.sumsq), self.stream)
            if all_dense:
                call("seqrec_sumsq", ptr(self.flat_g), self.flat_g.numel(), ptr(self.sumsq), st)
            else:
                for n, off, sz in segs:
                    if self.trainable[n]:
                        call("seqrec_sumsq", ptr(self.flat_g[off:off + sz]), sz, ptr(self.sumsq), st)
            self._join()
        adam = o["kind"] == "adam"
        with self._branch():
            if w.x_dense is None:
                if self.trainable["W_in"]:
                    # also re-zeroes the touched rows of dW_in and their flags (zero invariant of the dense buffer)
                    if adam:
                        self._adam_table(self.stream)
                    else:
                        call("seqrec_adagrad_rows", ptr(self.W_in), ptr(self.dW_in), ptr(self.aW_in), ptr(self.rows),
                             ptr(self.n_rows), ptr(self.touched), self.GH, max_rows, o["lr"], o["eps"], o["clipnorm"],
                             ptr(self.sumsq), den, self.stream)
                else:
                    self.dW_in.zero_()
                    self.touched.zero_()
            else:
                if self.trainable["W_in"]:
                    if adam:
                        self._adam(self.W_in, self.dW_in, self.mW_in, self.aW_in, self.stream)
                    else:
                        call("seqrec_adagrad", ptr(self.W_in), ptr(self.dW_in), ptr(self.aW_in), self.W_in.numel(),
                             o["lr"], o["eps"], o["clipnorm"], ptr(self.sumsq), den, self.stream)
                self.dW_in.zero_()
        if all_dense:
            if adam:
                self._adam(self.flat_p, self.flat_g, self.flat_m, self.flat_a, st)
            else:
                call("seqrec_adagrad", ptr(self.flat_p), ptr(self.flat_g), ptr(self.flat_a), self.flat_p.numel(),
                     o["lr"], o["eps"], o["clipnorm"], ptr(self.sumsq), den, st)
        else:
            for n, off, sz in segs:
                if self.trainable[n]:
                    if adam:
                        self._adam(self.flat_p[off:off + sz], self.flat_g[off:off + sz], self.flat_m[off:off + sz],
                                   self.flat_a[off:off + sz], st)
                    else:
                        call("seqrec_adagrad", ptr(self.flat_p[off:off + sz]), ptr(self.flat_g[off:off + sz]),
                             ptr(self.flat_a[off:off + sz]), sz, o["lr"], o["eps"], o["clipnorm"], ptr(self.sumsq),
                             den, st)
        self._join()
        if adam:
            self.iterations.add_(1)               # after both halves: each read the count of the updates before it

    def _adam(self, p, g, m, v, st):
        """Dense Adam over p (the flat buffer, one of its segments or the dense W_in of the x_dense input path)."""
        o = self.opt
        call("seqrec_adam", ptr(p), ptr(g), ptr(m), ptr(v), p.numel(), o["lr"], o["beta_1"], o["beta_2"], o["eps"],
             o["decay"], o["clipnorm"], ptr(self.sumsq), ptr(self.n_valid_f), ptr(self.iterations), st)

    def _adam_table(self, st):
        """Adam over every row of the W_in table; reads and re-zeroes only the touched rows of dW_in."""
        o = self.opt
        call("seqrec_adam_table", ptr(self.W_in), ptr(self.dW_in), ptr(self.mW_in), ptr(self.aW_in), ptr(self.touched),
             self.F, self.GH, o["lr"], o["beta_1"], o["beta_2"], o["eps"], o["decay"], o["clipnorm"], ptr(self.sumsq),
             ptr(self.n_valid_f), ptr(self.iterations), st)

    def _topk_rows(self, wt, k):
        """Top-k of the wt.N rows of wt.hout against THIS rank's items (ids are local item indices), probabilities from
        the softmax statistics (wt.m, wt.s)."""
        hrows, m, s, n = wt.hout, wt.m, wt.s, wt.N
        out_i = torch.empty((n, k), dtype=torch.int32, device=self.device)
        out_p = torch.empty((n, k), dtype=torch.float32, device=self.device)
        n_lists = wt.tc["splits"] if wt.tc["fwd"] else 0
        if wt.tc["fwd"] and k <= 32 and n_lists * k <= 384 and os.environ.get("SEQREC_TOPK_TC", "1") != "0":
            # tensor-core ranking: the bf16 hi/lo operands were staged by the statistics pass
            ws_v = torch.empty((n_lists, n, k), dtype=torch.float32, device=self.device)
            ws_i = torch.empty((n_lists, n, k), dtype=torch.int32, device=self.device)
            call("seqrec_topk_tc", ptr(wt.A_hi), ptr(wt.A_lo), ptr(self.Bt_hi), ptr(self.Bt_lo), ptr(self.b_out), ptr(m),
                 ptr(s), ptr(ws_v), ptr(ws_i), ptr(out_i), ptr(out_p), n, self.Hk, self.V, int(k),
                 1 if self.tc_x3 else 0, self.stream)
        else:
            call("seqrec_topk", ptr(hrows), ptr(self.W_out), ptr(self.b_out), ptr(m), ptr(s), ptr(out_i), ptr(out_p), n,
                 self.H, self.V, int(k), self.stream)
        return out_i, out_p

    def _topk_vp(self, w, k, last_step_only):
        """Vocabulary-parallel ranking (SURVEY 8(e)): all-gather the rows to score, every rank ranks them against its
        item shard with the catalog-wide softmax statistics, the P*k candidates of a row are gathered back and merged
        (probability descending, lower item id first on ties)."""
        comm = self.comm
        if k > self.V:
            raise ValueError("k must not exceed the items of one shard (%d)" % self.V)
        wg, _ = self._vp_gather(w, last_step_only, with_targets=False)
        n_loc = wg.N // comm.world
        self._vp_merge(wg, with_targets=False)                           # catalog-wide (m, s) of every gathered row
        loc_i, loc_p = self._topk_rows(wg, k)
        loc_i = loc_i + self.v_lo                                        # global item ids
        # every rank needs the P candidate lists of ITS rows only: one all-to-all (block j of the local result holds
        # rank j's rows), then the same (probability descending, lower id first) merge kernel the 1-GPU ranking ends with
        cand_i = comm.all_to_all_rows(loc_i)                             # (P lists, n_loc rows, k)
        cand_p = comm.all_to_all_rows(loc_p)
        if comm.world * k > 384:
            raise ValueError("vocabulary-parallel ranking needs world * k <= 384")
        top_i = torch.empty((n_loc, k), dtype=torch.int32, device=self.device)
        top_p = torch.empty((n_loc, k), dtype=torch.float32, device=self.device)
        call("seqrec_topk_merge", ptr(cand_p), ptr(cand_i), comm.world, n_loc * k, ptr(top_i), ptr(top_p), n_loc, k,
             self.stream)
        return top_i, top_p

    # ------------------------------------------------------------------------------------------------ gradients only
    def grad_batch(self, ids, tgt, x_dense=None, fused=None):
        """fwd + bwd WITHOUT the update (parity tests): returns loss and the raw (unclipped) gradients as numpy arrays
        in weight-list order.  Leaves the dW_in zero-invariant intact.  fused: None = what a training step runs."""
        B, T = (ids.shape if ids is not None else x_dense.shape[:2])
        w = self.work(int(B), int(T))
        st = self.stream
        saved_opt = self.opt
        self._stage(w, ids, tgt, x_dense, grads=True)
        self._forward_hidden(w, training=True)
        use_fused = (self.ce_fused if fused is None else bool(fused)) and w.tc["bwd"]
        if w.tc["panel"]:
            self._ce_panels(w, True, train=True, backward=True)
        elif use_fused:
            self._ce_train_fused(w)
        else:
            self._forward_ce(w, training=True, train=True)
        if not w.tc["panel"]:
            self._backward_ce(w, dh=not use_fused)
        dh = w.dh.clone()
        self._rnn_backward(w)
        self._rnn_weight_grad(w)
        if w.x_dense is None:
            call("seqrec_scatter_add_rows", ptr(w.xg), ptr(w.ids), ptr(w.mask), ptr(w.in_scale), ptr(self.dW_in),
                 ptr(self.touched), ptr(self.rows), ptr(self.n_rows), w.N, self.F, self.GH, st)
        else:
            self.dW_in.zero_()
            gemm(self, w.x_dense.view(w.N, self.F), w.xg.view(w.N, self.GH), self.dW_in, "tn")
        self.check_errors()
        # the kernels leave un-normalised gradients (the optimiser divides by n_valid): normalise here for the caller
        n_valid = float(self.n_valid_f.item())
        loss = float(self.step_loss_sum.item()) / n_valid
        grads = [self.dW_in, self.dU, self.db, self.dW_out] + ([self.db_out] if self.out_bias else [])
        out = [(g.detach().double() / n_valid).float().cpu().numpy() for g in grads]
        rows = self.rows[: int(self.n_rows.item())].cpu().numpy().copy() if w.x_dense is None else None
        self.dW_in.zero_()
        self.touched.zero_()
        self.opt = saved_opt
        return loss, out, dict(dh=(dh / n_valid).cpu().numpy(), rows=rows,
                               dxp=(w.xg.detach() / n_valid).cpu().numpy())

    # ------------------------------------------------------------------------------------------------ carried state
    def initial_state(self, n):
        """The zero state of n sessions: what every scan of a whole window starts from."""
        return RecurrentState.zeros(n, self.cell, self.H, self.device)

    def _state_operands(self, state, n):
        """(h0, c0) device pointers' tensors of a state of n sessions (c0 None unless LSTM)."""
        state.check(self.cell, self.H, n)
        h = state.h.to(self.device, torch.float32).contiguous()
        c = None if state.c is None else state.c.to(self.device, torch.float32).contiguous()
        return h, c

    def advance_state(self, ids, state=None, x_dense=None):
        """Continues the masked recurrence of a batch of sessions over a left-padded chunk of new events (B,T') and
        returns the state after it (fresh tensors).  state None = the zero state.  A pad step holds h and c, so an
        all-pad row keeps its state bit for bit; advancing by a and then by b equals advancing by a|b bit for bit."""
        w = self._scan_batch(ids, None, x_dense, state)
        return RecurrentState(w.hout[w.T - 1].clone(), w.cst[w.T - 1].clone() if self.cell == "LSTM" else None,
                              self.cell, self.H)

    def _state_work(self, state, tgt=None):
        """The (n, 1) work object of the last_step_only scorers with hout = state.h.  Every row is scored (a state
        always has a next item); with targets, a target < 0 is a pad (p = 1e-7, rank 0)."""
        h, _ = self._state_operands(state, len(state))
        wl = self.work(len(state), 1)
        wl.hout[0].copy_(h)
        wl.hscale = None
        if tgt is None:
            wl.mask.fill_(1)
        else:
            self._check_host_ids(None, tgt)
            t = torch.as_tensor(tgt).to(self.device, torch.int32).reshape(-1)
            if t.numel() != wl.B:
                raise ValueError("%d targets for %d sessions" % (t.numel(), wl.B))
            if bool((t >= self.V_total).any()):
                raise ValueError("target id outside the catalog (%d items)" % self.V_total)
            wl.tgt[0].copy_(t)
            wl.mask[0].copy_(t >= 0)
        return wl

    def topk_from_state(self, state, k):
        """Top-k next items after each session's state: (n,k) ids and probabilities, computed by the kernels of
        topk_batch(last_step_only=True)."""
        return self._topk_scored(self._state_work(state), int(k), True)

    def target_prob_from_state(self, state, tgt):
        """p(tgt[i] is the next item of session i), (n,) clipped like target_prob_batch."""
        return self._target_prob(self._state_work(state, tgt)).clone()

    def target_rank_from_state(self, state, tgt):
        """(n,) int32 rank of tgt[i] after session i's state, as target_rank_batch(last_step_only=True)."""
        return self._rank_scored(self._state_work(state, tgt), True)

    def candidates_from_state(self, state, cand, k=None, probs=False):
        """The candidate order after each session's state: (n,k) ids and scores, as candidates_batch(last_step_only=
        True).  cand (n, C)."""
        lists, k = self._candidate_lists(cand, (len(state),), k)
        return self._candidates_scored(self._state_work(state), lists, False, k, bool(probs), True)

    def candidate_rank_from_state(self, state, tgt, cand):
        """(n,) int32 rank of tgt[i] among session i's candidates cand[i] after its state."""
        lists, _ = self._candidate_lists(cand, (len(state),))
        return self._candidates_scored(self._state_work(state, tgt), lists, True, None, False, True)

    # ------------------------------------------------------------------------------------------------ scoring
    # Every scorer: stage the batch and scan (_scan_batch; the *_from_state scorers build their (n, 1) problem with
    # _state_work instead), score every step or the last one (_target_prob, _rank_scored, _topk_scored: the only places
    # that tell a vocabulary-parallel model from a replicated one), lay the time-major results out per session.
    def _scan_batch(self, ids, tgt, x_dense=None, initial_state=None):
        """Stages a (B,T) batch and runs the inference scan from initial_state (None = zeros); returns the work object."""
        B, T = (ids.shape if ids is not None else x_dense.shape[:2])
        w = self.work(int(B), int(T))
        self._stage(w, ids, tgt, x_dense)
        self._forward_hidden(w, training=False, state=initial_state)
        return w

    def _per_session(self, x, w):
        """Time-major results of w's tokens (N, ...) laid out per session, (B, T, ...), in storage of their own.  (When
        T or B is 1 the transposed view of a work buffer is contiguous already: .contiguous() would return the buffer.)"""
        x = x.view((w.T, w.B) + tuple(x.shape[1:])).transpose(0, 1)
        return x.clone(memory_format=torch.contiguous_format)

    def _last_step(self, w, with_targets=False):
        """The (B, 1) problem over the rows hout[T-1] of w (step T-1 of every session), with their mask and, when the
        call has targets, their targets."""
        wl = self.work(w.B, 1)
        if wl is not w:
            wl.hout.copy_(w.hout[w.T - 1:w.T])
            wl.mask.copy_(w.mask[w.T - 1:w.T])
            if with_targets:
                wl.tgt.copy_(w.tgt[w.T - 1:w.T])
        wl.hscale = None
        return wl

    def hidden_batch(self, ids, x_dense=None, initial_state=None):
        """(B,T,H) hidden outputs (z_to_z_output activations), inference phase."""
        w = self._scan_batch(ids, None, x_dense, initial_state)
        return self._per_session(w.hout.view(w.N, self.H), w)

    def predict_batch(self, ids, x_dense=None):
        """model.predict: (B,T,V) float32 softmax probabilities on the device."""
        if self.vocab_parallel:
            raise NotImplementedError("a vocabulary-parallel model never materialises (B,T,V): use topk_batch / "
                                      "target_prob_batch, or gather the weights into a replicated model")
        w = self._scan_batch(ids, None, x_dense)
        probs = torch.empty((w.B, w.T, self.V), dtype=torch.float32, device=self.device)
        if w.tc["panel"]:
            # hidden sizes above 256: logits through the plain GEMM (model.predict materialises (N,V) by definition)
            Z, m, s_ = self._wide_logits(w.hout.view(w.N, self.H))
            call("seqrec_softmax_rows_probs", ptr(Z), ptr(m), ptr(s_), ptr(probs), w.T, w.B, self.V, self.stream)
            return probs
        self._forward_ce(w, with_targets=False)
        call("seqrec_predict_probs", ptr(w.hout), ptr(self.W_out), ptr(self.b_out), ptr(w.m), ptr(w.s), ptr(probs),
             w.T, w.B, self.H, self.V, self.stream)
        return probs

    def target_prob_batch(self, ids, tgt, x_dense=None, initial_state=None):
        """p(true next item) per step, clipped to [1e-7, 1-1e-7] like model.py:108-110; (B,T) device tensor.
        initial_state: the sessions' RecurrentState the chunk continues (None = zeros)."""
        w = self._scan_batch(ids, tgt, x_dense, initial_state)
        return self._per_session(self._target_prob(w), w)

    def _target_prob(self, w):
        """(N,) p(target) of w's tokens, time-major (a view of a work buffer)."""
        if self.vocab_parallel:
            # every rank scores all ranks' tokens against its item shard; the merged statistics cover the whole catalog
            return self._my_rows(self._vp_forward(w, training=False).py)
        self._forward_ce(w)
        return w.py

    # ------------------------------------------------------------------------------------------------ target rank
    def _stage_rows_operands(self, w):
        """bf16 hi/lo operands of the tensor-core logits pass for the rows of w.hout (inference: no dropout factors)."""
        self._stage_weight_operands()
        call("seqrec_split_bf16", ptr(w.hout), None, ptr(w.A_hi), ptr(w.A_lo), w.N, self.H, self.Hk, 0, self.stream)
        w.tc_operands_fresh = True

    def _rank_rows_count(self, w, ref, rank, id_offset):
        """Adds to rank[n] the number of THIS model's items that precede the target w.tgt[n] (a global id) in the stable
        descending logit order, for the N rows of w.hout.  ref: per-token reference logit (None: the SIMT kernel computes
        z_y itself with the arithmetic of every z_v).  The tensor-core pass also leaves the softmax partials of the rows
        in w.ws_m / w.ws_s; returns their number of rows (0 on the SIMT kernel, which computes no statistics)."""
        st = self.stream
        if w.tc["fwd"]:
            self._stage_rows_operands(w)
            call("seqrec_ce_tc_forward_rank", ptr(w.A_hi), ptr(w.A_lo), ptr(self.Bt_hi), ptr(self.Bt_lo),
                 ptr(self.b_out), ptr(w.ws_m), ptr(w.ws_s), ptr(ref), ptr(w.tgt), int(id_offset), ptr(rank), w.N,
                 self.Hk, self.V, 0, self.V, 1 if self.tc_x3 else 0, st)
            return w.tc["splits"]
        call("seqrec_target_rank", ptr(w.hout), ptr(self.W_out), ptr(self.b_out), ptr(ref), ptr(w.tgt), int(id_offset),
             ptr(rank), w.N, self.H, self.V, 0, self.V, self.V, st)
        return 0

    def _target_rank(self, w):
        """(N,) int32 1-based rank of w.tgt in the logits of w.hout's rows, 0 on pads."""
        st = self.stream
        N = w.N
        tg = w.tgt.view(-1)
        if w.tc["panel"]:
            # hidden sizes above 256: panels of materialised logits (never the (N,V) matrix), ranked row by row
            rank = torch.empty(N, dtype=torch.int32, device=self.device)
            nb_max = max(128, ((256 << 20) // (4 * self.V)) // 128 * 128)
            rows = w.hout.view(N, self.H)
            Z = torch.empty((min(nb_max, N), self.V), dtype=torch.float32, device=self.device)
            for n0 in range(0, N, nb_max):
                nb = min(nb_max, N - n0)
                gemm(self, rows[n0:n0 + nb], self.W_out, Z[:nb], "nn", bias=self.b_out)
                call("seqrec_rows_rank", ptr(Z[:nb]), ptr(tg[n0:n0 + nb]), ptr(rank[n0:n0 + nb]), nb, self.V, st)
            return rank
        rank = (tg >= 0).to(torch.int32)                 # the 1 of the 1-based rank; the kernels add the count
        if w.tc["fwd"]:
            # the exact fp32 target logit is the reference of the count: it must be complete BEFORE the pass (the
            # statistics pass overlaps it, because there it is only needed by the finalize kernel)
            call("seqrec_target_logit", ptr(w.hout), None, ptr(self.W_out), ptr(self.b_out), ptr(w.tgt), ptr(w.zy), N,
                 self.H, self.V, None, None, st)
            n_splits = self._rank_rows_count(w, w.zy, rank, 0)
            # the pass wrote the softmax partials too: p(target) of the same rows comes for one finalize kernel
            self._finalize_ce(w, w.ws_m, w.ws_s, n_splits)
        else:
            self._rank_rows_count(w, None, rank, 0)
        return rank

    def _rank_vp(self, w, last_step_only):
        """Vocabulary-parallel rank: every rank counts, for all ranks' rows, the items of ITS shard that precede the
        target (global ids, id_offset = the shard's first item) against the catalog-wide reference logit (computed on
        the target's owner shard, summed over the shards); the integer counts are summed over the shards."""
        comm = self.comm
        wg, tgt_all = self._vp_gather(w, last_step_only)
        call("seqrec_target_logit", ptr(wg.hout), None, ptr(self.W_out), ptr(self.b_out), ptr(wg.tgt), ptr(wg.zy),
             wg.N, self.H, self.V, None, None, self.stream)
        comm.all_reduce_sum(wg.zy)                        # only the owner shard contributes: the exact fp32 z_y
        wg.tgt.view(-1).copy_(tgt_all)                    # global ids from here on
        counts = torch.zeros(wg.N, dtype=torch.int32, device=self.device)
        self._rank_rows_count(wg, wg.zy, counts, self.v_lo)
        comm.all_reduce_sum(counts)
        return self._my_rows(counts) + (self._my_rows(tgt_all) >= 0).to(torch.int32)

    def target_rank_batch(self, ids, tgt, x_dense=None, last_step_only=False, initial_state=None):
        """Rank of the true next item per step: (B,T) int32 device tensor, or (B,) for the last step only.
        rank = 1 + #{v != y : z_v > z_y} + #{v < y : z_v == z_y} (stable descending order, ties to the lower item id:
        rank <= k <=> topk_batch holds y at index rank-1); pads have rank 0.  On the tensor cores the logits are compared
        with the exact fp32 target logit, so the rank is exact outside the band of the split-product error around z_y,
        and p(target) of the same rows is left in the work object's `py` by the same pass.
        initial_state: the sessions' RecurrentState the chunk continues (None = zeros)."""
        w = self._scan_batch(ids, tgt, x_dense, initial_state)
        return self._rank_scored(w, last_step_only)

    def _rank_scored(self, w, last_step_only):
        """Target ranks of every step of w, (B,T), or of its last step, (B,)."""
        if self.vocab_parallel:
            rank = self._rank_vp(w, last_step_only)
        else:
            rank = self._target_rank(self._last_step(w, with_targets=True) if last_step_only else w)
        return rank if last_step_only else self._per_session(rank, w)

    def _wide_logits(self, rows):
        """Hidden sizes above 256: logits of `rows` (n, H) materialised through the plain GEMM (tcgen05 when it fills
        tiles) with their per-row softmax statistics.  Scoring helper: n is a batch of rows, never the training set."""
        n = rows.shape[0]
        Z = torch.empty((n, self.V), dtype=torch.float32, device=self.device)
        gemm(self, rows.contiguous(), self.W_out, Z, "nn", bias=self.b_out)
        m = torch.empty(n, dtype=torch.float32, device=self.device)
        s_ = torch.empty(n, dtype=torch.float32, device=self.device)
        call("seqrec_softmax_rows_stats", ptr(Z), None, ptr(m), ptr(s_), None, n, self.V, self.stream)
        return Z, m, s_

    def topk_batch(self, ids, k, last_step_only=True, x_dense=None, initial_state=None):
        """Top-k next items: (B,k) ids and probabilities for the last step, or (B,T,k) for every step.
        initial_state: the sessions' RecurrentState the chunk continues (None = zeros)."""
        w = self._scan_batch(ids, None, x_dense, initial_state)
        return self._topk_scored(w, int(k), last_step_only)

    def _topk_scored(self, w, k, last_step_only):
        """Top-k of the rows of w.hout (all steps, or the last one)."""
        if self.vocab_parallel:
            top_i, top_p = self._topk_vp(w, k, last_step_only)
        else:
            wt = self._last_step(w) if last_step_only else w
            if wt.tc["panel"]:
                Z, m, s_ = self._wide_logits(wt.hout.view(wt.N, self.H))
                order = torch.sort(Z, dim=1, descending=True, stable=True)      # ties: the lower item id first
                top_i = order.indices[:, :k].to(torch.int32).contiguous()
                top_p = (torch.exp(order.values[:, :k] - m.unsqueeze(1)) / s_.unsqueeze(1)).contiguous()
            else:
                # softmax statistics of the rows to rank (the last step: a (B, 1) problem over the rows hout[T-1])
                self._forward_ce(wt, with_targets=False)
                top_i, top_p = self._topk_rows(wt, k)
        if last_step_only:
            return top_i, top_p
        return self._per_session(top_i, w), self._per_session(top_p, w)

    # ------------------------------------------------------------------------------------------------ candidates
    def candidates_batch(self, ids, cand, k=None, probs=False, last_step_only=True, x_dense=None, initial_state=None):
        """Scores a given candidate list per session: cand (B, C) for the last step, (B, T, C) for every step; ids < 0
        are pads.  Returns (ids int32, scores float32) of the first k (default C) entries of the order -- score
        descending, then lower item id, then lower list position, pads last as (-1, 0) -- of shape (B, k) or (B, T, k).
        Scores are the logits, or with probs=True the catalog softmax probabilities (one statistics pass).
        initial_state: the sessions' RecurrentState the chunk continues (None = zeros)."""
        B, T = (ids.shape if ids is not None else x_dense.shape[:2])
        lists, k = self._candidate_lists(cand, (int(B),) if last_step_only else (int(B), int(T)), k)
        w = self._scan_batch(ids, None, x_dense, initial_state)
        return self._candidates_scored(w, lists, False, k, bool(probs), last_step_only)

    def candidate_rank_batch(self, ids, tgt, cand, last_step_only=False, x_dense=None, initial_state=None):
        """Rank of the true next item among the candidates, (B,T) int32 (cand (B, T, C)) or (B,) for the last step
        (cand (B, C)): 1 + #{j : c_j >= 0, c_j != y, z_j > z_y or (z_j == z_y and c_j < y)}; 0 where y < 0."""
        B, T = (ids.shape if ids is not None else x_dense.shape[:2])
        lists, _ = self._candidate_lists(cand, (int(B),) if last_step_only else (int(B), int(T)))
        w = self._scan_batch(ids, tgt, x_dense, initial_state)
        return self._candidates_scored(w, lists, True, None, False, last_step_only)

    def _candidate_lists(self, cand, lead, k=None):
        """Validated candidate lists as a contiguous device int32 tensor (every id < 0 becomes the pad -1), and k."""
        cand, _, k = check_candidates(cand, lead, self.V_total, k)
        t = cand if isinstance(cand, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(cand))
        return t.to(self.device).clamp(min=-1).to(torch.int32).contiguous(), k

    def _stage_item_major(self):
        """fp32 W_out^T (V, H): the candidate logits read one coalesced row per item instead of a strided column of
        W_out.  Made on first use and again whenever the weights changed; V*H*4 bytes."""
        if self._wt_version != self._w_version:
            if self.Wt_items is None:
                self.Wt_items = torch.empty((self.V, self.H), dtype=torch.float32, device=self.device)
            call("seqrec_transpose", ptr(self.W_out), ptr(self.Wt_items), self.H, self.V, self.stream)
            self._wt_version = self._w_version
        return self.Wt_items

    def _candidate_logits(self, rows, lists, id_offset):
        """(n, C) logits of the lists (n, C) of global ids against this model's items (0 for pads and other shards)."""
        n, C = lists.shape
        z = torch.empty((n, C), dtype=torch.float32, device=self.device)
        call("seqrec_candidate_logits", ptr(rows), ptr(self._stage_item_major()), ptr(self.b_out), ptr(lists), C, ptr(z),
             n, C, self.H, int(id_offset), self.V, self.stream)
        return z

    def _candidates_scored(self, w, cand, tgt, k, probs, last_step_only):
        """Candidate scoring of the rows of w.hout (all steps, or the last one).  cand: device int32 lists, (B, C) or
        (B, T, C).  tgt True: the ranks of w's staged targets among them, (B,) or (B,T); else the first k entries of the
        order, (ids, scores), with catalog probabilities when probs.  With a target the list is [y | candidates], so z_y
        comes from the candidate arithmetic (and, on a vocabulary shard, from the same reduction)."""
        C = cand.shape[-1]
        lists = cand if last_step_only else cand.transpose(0, 1).reshape(w.N, C)       # time-major rows
        m = s = None
        if self.vocab_parallel:
            comm = self.comm
            y = (w.tgt[w.T - 1] if last_step_only else w.tgt.view(-1)) if tgt else None
            scored = torch.cat([y[:, None], lists], 1) if tgt else lists
            wg, _ = self._vp_gather(w, last_step_only, with_targets=False)
            part = self._candidate_logits(wg.hout.view(wg.N, self.H), comm.all_gather_cat(scored), self.v_lo)
            Z = torch.empty(scored.shape, dtype=torch.float32, device=self.device)
            comm.reduce_scatter_sum(Z, part)                 # one non-zero addend per entry: the owner shard's logit
            if probs:
                self._vp_merge(wg, with_targets=False)
                m, s = self._my_rows(wg.m), self._my_rows(wg.s)
        else:
            wt = self._last_step(w, with_targets=tgt) if last_step_only else w
            rows = wt.hout.view(wt.N, self.H)
            y = wt.tgt.view(-1) if tgt else None
            Z = self._candidate_logits(rows, torch.cat([y[:, None], lists], 1) if tgt else lists, 0)
            if probs:
                if wt.tc["panel"]:
                    _, m, s = self._wide_logits(rows)
                else:
                    self._forward_ce(wt, with_targets=False)
                    m, s = wt.m, wt.s
        n = lists.shape[0]
        if tgt:
            rank = torch.empty(n, dtype=torch.int32, device=self.device)
            z, zy = Z[:, 1:].contiguous(), Z[:, 0].contiguous()
            call("seqrec_candidate_order", ptr(z), ptr(lists), C, n, None, None, 0, None, None, ptr(zy), ptr(y),
                 ptr(rank), self.stream)
            return rank if last_step_only else self._per_session(rank, w)
        out_i = torch.empty((n, k), dtype=torch.int32, device=self.device)
        out_s = torch.empty((n, k), dtype=torch.float32, device=self.device)
        call("seqrec_candidate_order", ptr(Z), ptr(lists), C, n, ptr(m), ptr(s), k, ptr(out_i), ptr(out_s), None, None,
             None, self.stream)
        if last_step_only:
            return out_i, out_s
        return self._per_session(out_i, w), self._per_session(out_s, w)
