#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json: training sequences/sec, % of roofline, vs CPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one synthetic batch: item-row gather, recurrent scan, fused logits +
softmax-CE, backward (incl. the embedding-gradient scatter-add), global-norm clip and Adagrad -- plus the gradient
all-reduce when N > 1 (weak scaling: every rank owns B sequences).  Workload at N=1: configs[1] of BASELINE.json
(Reddit-like: V=10k, GRU-128, T=50, B=256).  Rank 0 prints ONE JSON line.

Timing: W warm-up steps, then K steps each bracketed by CUDA events on the launching stream, an L2 flush (a 256 MiB
memset, outside the events) between steps, barrier + synchronize on both sides, max over ranks.

--dump-outputs DIR writes what the headline workload's last timed step returned to its caller as DIR/<name>.npy
(float32; item ids as float64), at most 64 MiB in all, so that two builds can be compared output for output on the
same seeded inputs.  Training: the step's loss and the weights after it (U and b whole; the rows of W_in and the
columns of W_out of a fixed item sample, DIR/sample_items.npy).  Scoring (cfg5): the top-k ids and probabilities of
the last step and p(true next item) at every step.  Gradient sums are accumulated with atomics, so two runs of the same
build differ slightly: compare with a tolerance.  Measured on a B200 at 1000 W, cfg4, 20 steps: loss to 1.3e-7
relative, W_out to 1.2e-5, b to 2.7e-4, U to 7.3e-4, W_in rows to 2.2e-3.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "training sequences/sec"
DEFAULT_CONFIG = "cfg4_gru256_1m"
DUMP_SAMPLE_ITEMS = 8192
DUMP_SAMPLE_BYTES = 48 << 20           # item-indexed weight slices; U and b add at most a few MiB on top


def save_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype.kind in "iu" else np.float32))


def sample_items(V, n, seed=0):
    """The items whose W_in rows / W_out columns --dump-outputs writes: the n/2 lowest ids (the most frequent under
    the Zipf workload, so rows that every step updates) and a seeded uniform draw of n/2 from the rest."""
    if V <= n:
        return np.arange(V, dtype=np.int64)
    rng = np.random.default_rng(seed)
    tail = n // 2 + rng.choice(V - n // 2, size=n - n // 2, replace=False)
    return np.sort(np.concatenate([np.arange(n // 2), tail])).astype(np.int64)


def dump_training_outputs(hot, loss, out_dir, rank):
    """The loss of the last timed step and the weights it left.  Under vocabulary parallelism every rank contributes
    the sampled W_out columns of its own shard (one all-reduce of an (H, n) block), so every rank must call; rank 0
    writes."""
    import torch
    n = min(DUMP_SAMPLE_ITEMS, max(1, DUMP_SAMPLE_BYTES // (4 * (hot.GH + hot.H))))
    items = sample_items(hot.V_total, n)
    idx = torch.from_numpy(items).to(hot.device)
    own = (idx >= hot.v_lo) & (idx < hot.v_lo + hot.V)
    cols = torch.zeros((hot.H, len(items)), dtype=torch.float32, device=hot.device)
    cols[:, own] = hot.W_out.index_select(1, idx[own] - hot.v_lo)
    if hot.vocab_parallel:
        hot.comm.all_reduce_sum(cols)
    arrays = {"loss": loss.detach().float().cpu().numpy(), "sample_items": items,
              "W_in_rows": hot.W_in.index_select(0, idx).cpu().numpy(), "U": hot.U.cpu().numpy(),
              "b": hot.b.cpu().numpy(), "W_out_cols": cols.cpu().numpy()}
    if rank == 0:
        save_outputs(out_dir, arrays)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


def load_traffic(workload, prefix="ce_tc_backward"):
    """(bytes, detail): dram__bytes_read.sum + dram__bytes_write.sum of the dominant phase -- the kernels whose name starts
    with `prefix`, one launch each per call of seqrec_ce_tc_backward -- from the committed ncu --set full capture of this
    workload (profiles/traffic.json, written by scripts/summarize_ncu.py), and the per-kernel entries behind the sum;
    (None, None) when the workload was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            detail = json.load(f).get(workload)
        dom = [v["dram_bytes_per_launch"] for k, v in detail.items() if k.startswith(prefix)]
        return (float(sum(dom)) if dom else None), detail
    except Exception:
        return None, None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the run: an NVML polling thread (5 ms period) when nvidia_ml_py is
    importable, else `nvidia-smi -lms 100` in a subprocess.  stop() reports the median clock under load."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        import threading
        self.sm, self.mx, self.reasons = [], [], set()
        self.p = self.f = self.thread = None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))

            def poll():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        try:
                            bits = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            bits = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for n, bit in self.REASONS.items():
                            if bits & bit:
                                self.reasons.add(n)
                    except Exception:
                        pass
                    self._stop.wait(0.005)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark(self):
        """Samples taken before this call are dropped (start of the timed region)."""
        if self.thread is not None:
            del self.sm[:]
            self.reasons.clear()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            out["source"] = "nvml"
        elif self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush()
            self.f.seek(0)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for line in self.f.read().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    self.sm.append(float(c[1]))
                    self.mx.append(float(c[2]))
                except ValueError:
                    continue
                for n, v in zip(names, c[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            os.unlink(self.f.name)
            out["source"] = "nvidia-smi"
        if self.sm:
            out["sm_mhz"] = float(np.median(self.sm))
            out["sm_max_mhz"] = float(max(self.mx)) if self.mx else None
            out["samples"] = len(self.sm)
        out["reasons"] = sorted(self.reasons)
        return out


def algorithmic_work(cfg, n_tokens):
    """SURVEY §8(d) per-unit figures x the units one launch processes."""
    G = {"simpleRNN": 1, "LSTM": 4, "GRU": 3}[cfg["cell"]]
    H, V = cfg["H"], cfg["V"]
    GH = G * H
    return {
        "gather_bytes": n_tokens * (4 + 2 * GH * 4),
        "scatter_bytes": n_tokens * (4 + 3 * GH * 4),
        "rnn_fwd_flops": n_tokens * 2 * G * H * H,
        "rnn_bwd_flops": n_tokens * 4 * G * H * H,
        "ce_fwd_flops": n_tokens * 2 * H * V,
        "ce_bwd_flops": n_tokens * 4 * H * V,
        "step_flops": n_tokens * (6 * G * H * H + 6 * H * V),
    }


# ------------------------------------------------------------------------------------------------------------------
def cpu_oracle_step_fn(cfg, ids, tgt, seed):
    """The oracle port (torch-CPU fp32 restatement of the Keras/Theano arithmetic) -- the CPU baseline."""
    import torch
    from oracle import keras_semantics as ks
    from seq_recommendations_b200 import synthetic
    ws = synthetic.make_weights(cfg["cell"], cfg["V"], cfg["H"], seed=seed)
    ora = ks.Model(cfg["cell"], cfg["act"], ws, dtype=torch.float32)
    ti, tt = torch.tensor(ids.astype(np.int64)), torch.tensor(tgt.astype(np.int64))
    mask = ti >= 0

    def step():
        loss, _, _ = ora.train_step(ti, tt, mask, lr=0.01, epsilon=1e-8, clipnorm=1.0)
        return float(loss)
    return step


def time_cpu(cfg, steps, warmup, budget_s=None, sample_b=None):
    """The oracle port timed on the host cores, `steps` steps at every timed batch size (fewer only when a budget_s in
    seconds is given and runs out; `timed_steps` reports the counts).  When the workload's batch fits (sample_b == B)
    the median step time is the result.  Otherwise (cfg3 / cfg4: the (N, V) logits of the full batch do not fit host
    memory) the step time is fitted as t(B) = a + b*B on two reduced batches -- the reference updates the whole
    (V, G*H) table densely every step, a cost that does not shrink with the batch -- and the value is
    B_full / t(B_full)."""
    import torch
    from seq_recommendations_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B_full = cfg["B"]
    sample_b = sample_b or B_full

    def median_step_ms(B, n_steps, n_warm, budget):
        ids, tgt = synthetic.make_batch(cfg["V"], cfg["T"], B, seed=0)
        step = cpu_oracle_step_fn(cfg, ids, tgt, seed=0)
        for _ in range(n_warm):
            step()
        times = []
        t_all = time.perf_counter()
        for _ in range(n_steps):
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
            if budget is not None and time.perf_counter() - t_all > budget:
                break
        return float(np.median(times)) * 1e3, len(times)

    if sample_b >= B_full:
        ms, n = median_step_ms(B_full, steps, warmup, budget_s)
        return dict(value=B_full / (ms / 1e3), unit="sequences/sec", cores=torch.get_num_threads(), kind="port",
                    sample="%d steps of fwd+bwd+clip+Adagrad on B=%d,T=%d,V=%d (oracle/keras_semantics.py, torch-CPU "
                           "fp32, median)" % (n, B_full, cfg["T"], cfg["V"]), ms_per_step=ms, timed_steps=[n])
    b1, b2 = max(1, sample_b // 2), max(2, sample_b // 2 * 3)
    half = None if budget_s is None else budget_s / 2
    ms1, n1 = median_step_ms(b1, steps, min(warmup, 1), half)
    ms2, n2 = median_step_ms(b2, steps, 0, half)
    slope = max((ms2 - ms1) / (b2 - b1), 0.0)
    fixed = max(ms1 - slope * b1, 0.0)
    ms = fixed + slope * B_full
    return dict(value=B_full / (ms / 1e3), unit="sequences/sec", cores=torch.get_num_threads(), kind="port",
                sample="fwd+bwd+clip+Adagrad (oracle/keras_semantics.py, torch-CPU fp32) at T=%d,V=%d on B=%d (%.0f ms, "
                       "%d steps) and B=%d (%.0f ms, %d steps); t(B) = %.0f ms + %.1f ms*B extrapolated to B=%d" % (
                           cfg["T"], cfg["V"], b1, ms1, n1, b2, ms2, n2, fixed, slope, B_full), ms_per_step=ms,
                timed_steps=[n1, n2])


def scan_info(cfg, B):
    """Wave structure of the tensor-core recurrent scan for this shape on THIS device: a cluster owns 64 batch rows for
    all timesteps, and the part keeps only `clusters_resident` of them on its SMs at once (GPC geometry;
    cudaOccupancyMaxActiveClusters) -- more row groups than that run as a second wave.  None when the shape runs on the
    register / generic scans."""
    from seq_recommendations_b200 import _lib
    cell = _lib.CELL.get(cfg["cell"], -1)
    lib = _lib.load()
    if cell < 0 or not lib.seqrec_rnn_tc_applicable(cell, cfg["H"]) or not (cfg["H"] > 128 or cfg["cell"] == "LSTM"):
        return None                                # (GRU-128 stays on the register scan: engine.HotPath.rnn_tc)
    resident = int(lib.seqrec_rnn_tc_max_clusters(cell, cfg["H"]))
    needed = (B + 63) // 64
    return {"kernel": "rnn_tc_*_kernel", "rows_per_cluster": 64, "cluster_size": cfg["H"] // 32,
            "clusters_needed": needed, "clusters_resident": resident,
            "waves": (needed + resident - 1) // resident if resident > 0 else None}


def config_dict(args, name, cfg, world, B, vp, cuda_graph):
    """The `config` object of the JSON line -- ONE function for both arms, so the driver's same-config check compares
    like with like."""
    return {"workload": name, "cell": cfg["cell"], "act": cfg["act"], "V": cfg["V"], "H": cfg["H"], "T": cfg["T"],
            "B_per_gpu": B, "global_batch": world * B,
            "parallelism": ("dp%d x vocab-parallel logits (W_out column-sharded)" % world) if vp else "dp%d" % world,
            "l2": "256 MiB memset between timed steps (outside the events)", "dropout": args.dropout,
            "optimizer": "adagrad lr=0.01 eps=1e-8 clipnorm=1", "cuda_graph": cuda_graph}


def cpu_sample_batch(cfg, B):
    """Bounded CPU sample: the batch is scaled down until the (N, V) logits of one oracle step hold about 2e8 elements
    (a second or so per step on the box's cores); sequences/sec is linear in B at fixed T and V."""
    return B if cfg["V"] * B * cfg["T"] <= 2e8 else max(1, int(2e8 // (cfg["V"] * cfg["T"])))


def run_reference(args, cfg, name):
    """--impl reference: the reference's CPU path on this arm's config.  The reference itself (Python 2 + Keras 2.0.x +
    Theano) cannot run in this image, so the oracle port stands in (DESIGN.md); every step is a bounded sample of the
    workload (cpu_sample_batch), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    sample_b = cpu_sample_batch(cfg, cfg["B"])
    r = time_cpu(cfg, args.steps, max(1, min(args.warmup, 2)), sample_b=sample_b)
    vp = (args.vocab_parallel == 1 or (args.vocab_parallel < 0 and name.startswith("cfg4"))) and world > 1 \
        and cfg["V"] % world == 0
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "sequences/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, name, cfg, world, cfg["B"], vp, True),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "timed_steps")},
        "e2e": {"value": r["value"], "unit": "sequences/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
def run_scoring(args, cfg, name, dump=None):
    """configs[4] (inference): sequences scored per second -- recurrent scan over T steps, then top-k next items of the
    last step (`last`) or p(true next item) at every step (`all`).  One step = one batch of B sequences.  dump: the
    directory --dump-outputs writes the last timed step's results to."""
    import torch
    from seq_recommendations_b200 import _lib
    from seq_recommendations_b200.engine import HotPath
    from seq_recommendations_b200 import synthetic
    torch.cuda.set_device(0)
    V, H, T, B, k = cfg["V"], cfg["H"], cfg["T"], cfg["B"], 20
    ws = synthetic.make_weights(cfg["cell"], V, H, seed=0)
    hot = HotPath(cfg["cell"], cfg["act"], V, H, V, weights=ws, tc=args.tc)
    ids, tgt = synthetic.make_batch(V, T, B, seed=0)
    pin_i, pin_t = torch.from_numpy(ids).pin_memory(), torch.from_numpy(tgt).pin_memory()
    dev_i, dev_t = pin_i.cuda(), pin_t.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out, results = {}, {}
    clocks = ClockSampler(0)
    for mode in ("last", "all"):
        run = (lambda i, t: hot.topk_batch(i, k, last_step_only=True)) if mode == "last" else (
            lambda i, t: (hot.target_prob_batch(i, t),))
        fn = lambda i, t: run(i, t)[0]
        for _ in range(max(args.warmup, 3)):
            fn(dev_i, dev_t)
        torch.cuda.synchronize()
        if mode == "last":
            clocks.mark()
        evs = []
        _lib.launch_count(reset=True)
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last = run(dev_i, dev_t)
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        launches = _lib.launch_count()
        if dump:
            names = ("top_items", "top_probs") if mode == "last" else ("target_probs",)
            results.update((n, r.cpu().numpy()) for n, r in zip(names, last))
        ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
        e2e = []
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn(pin_i, pin_t)
            r.cpu()
            e2e.append(time.perf_counter() - t0)
        out[mode] = dict(ms=ms, e2e_ms=float(np.mean(e2e)) * 1e3, launches=launches, d2h=int(r.numel() * r.element_size()))
    clk = clocks.stop()
    if dump:
        save_outputs(dump, results)
    peaks = load_peaks()
    G = 3 if cfg["cell"] == "GRU" else 4
    flops_all = B * T * (2 * G * H * H + 2 * H * V)
    line = {
        "metric": "sequences scored/sec", "value": B / (out["last"]["ms"] * 1e-3), "unit": "sequences/sec", "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": out["last"]["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 (bf16x3 split tensor-core GEMMs)" if hot.tc_x3 else hot.tc_mode,
        "data": "synthetic",
        "config": {"workload": name, "cell": cfg["cell"], "V": V, "H": H, "T": T, "B": B, "k": k,
                   "mode": "top-%d next items of the last step" % k,
                   "l2": "256 MiB memset between timed steps (outside the events)"},
        "clocks": clk,
        "e2e": {"value": B / (out["last"]["e2e_ms"] * 1e-3), "unit": "sequences/sec", "ms_per_step": out["last"]["e2e_ms"],
                "h2d_bytes_per_step": B * T * 4, "d2h_bytes_per_step": out["last"]["d2h"],
                "api": "HotPath.topk_batch(pinned host ids, k, last_step_only=True) -> ids.cpu()"},
        "gpu_launches": out["last"]["launches"],
        "scan": scan_info(cfg, B),
        "all_steps_target_prob": {"value": B / (out["all"]["ms"] * 1e-3), "unit": "sequences/sec",
                                  "ms_per_step": out["all"]["ms"], "e2e_ms_per_step": out["all"]["e2e_ms"],
                                  "algorithmic_tflops": flops_all / (out["all"]["ms"] * 1e-3) / 1e12,
                                  "frac_of_bf16_sustained": flops_all / (out["all"]["ms"] * 1e-3) / 1e12 / peaks["bf16_sustained"]},
        "roofline": {"kernel": "seqrec_ce_tc_forward over all B*T tokens (all-steps mode)", "bound": "tensor",
                     "achieved": flops_all / (out["all"]["ms"] * 1e-3) / 1e12, "peak": peaks["bf16_sustained"],
                     "unit": "TFLOP/s", "frac": flops_all / (out["all"]["ms"] * 1e-3) / 1e12 / peaks["bf16_sustained"],
                     "traffic": None},
        "cpu_baseline": None,
    }
    del hot, flush
    torch.cuda.empty_cache()
    return line


def measure_training(args, name, cfg, comm, rank, local, steps, warmup, full=True, batch=None, vp=None, dump=None):
    """One training workload on this process group: K timed steps with resident inputs (CUDA events, L2 flush between
    steps, barrier + synchronize on both sides, max over ranks), the same steps once more with an event at every phase
    boundary (per-kernel times), and the end-to-end leg from pinned host buffers.  `full` adds the reference-facing
    plugin leg, the CPU baseline and the clock sampler; `dump` is the directory the last timed step's outputs go to.
    Returns the JSON fields of this workload (rank 0) or None."""
    import torch
    from seq_recommendations_b200 import _lib, synthetic
    from seq_recommendations_b200.engine import HotPath

    world = comm.world
    dev = torch.device("cuda", local)
    V, H, T = cfg["V"], cfg["H"], cfg["T"]
    B = int(batch or cfg["B"])
    ws = synthetic.make_weights(cfg["cell"], V, H, seed=0)
    if vp is None:
        vp = (args.vocab_parallel == 1 or (args.vocab_parallel < 0 and name.startswith("cfg4"))) and world > 1 \
            and V % world == 0
    hot = HotPath(cfg["cell"], cfg["act"], V, H, V, weights=ws, comm=comm, seed=rank, tc=args.tc, vocab_parallel=vp)
    del ws
    hot.set_optimizer("adagrad", lr=0.01, epsilon=1e-8, clipnorm=1.0)
    hot.dropout_out = args.dropout
    n_batches = 4
    host = [synthetic.make_batch(V, T, B, seed=100 * rank + i) for i in range(n_batches)]
    pinned = [(torch.from_numpy(i).pin_memory(), torch.from_numpy(t).pin_memory()) for i, t in host]
    resident = [(i.to(dev), t.to(dev)) for i, t in pinned]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync_all():
        comm.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (the clock sampler is already running; its samples are reset when the timed region starts)
    clocks = ClockSampler(local) if rank == 0 else None
    for s in range(warmup):
        hot.train_batch(*resident[s % n_batches])
    sync_all()

    # ---- timed: K steps, inputs resident in HBM (the step replays as one CUDA graph)
    evs = []
    sync_all()
    if clocks is not None:
        clocks.mark()
    t_wall = time.perf_counter()
    for s in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = hot.train_batch(*resident[s % n_batches])
        e1.record()
        evs.append((e0, e1))
    sync_all()
    wall_s = time.perf_counter() - t_wall
    step_ms = sum(a.elapsed_time(b) for a, b in evs) / steps
    final_loss = float(loss.item())
    if dump:
        dump_training_outputs(hot, loss, dump, rank)
    hot.check_errors()
    # ---- the same K steps once more, launched eagerly with an event at every phase boundary: per-kernel times for the
    #      roofline and the launch count (a graph replay runs exactly these launches)
    graphs = hot.use_graphs
    hot.use_graphs = False
    _lib.launch_count(reset=True)
    hot.prof = []
    for s in range(steps):
        flush.zero_()
        hot.train_batch(*resident[s % n_batches])
    sync_all()
    launches = _lib.launch_count()
    phases = hot.phase_times_ms()
    hot.prof = None
    hot.use_graphs = graphs
    t = torch.tensor([step_ms], dtype=torch.float64, device=dev)
    comm.all_reduce_max(t)
    step_ms = float(t.item())

    # ---- e2e: same step through the public call with HOST buffers (pinned H2D of ids/targets + D2H of the loss)
    for s in range(3):
        float(hot.train_batch(*pinned[s % n_batches]).item())
    sync_all()
    e2e_t = []
    for s in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        float(hot.train_batch(*pinned[s % n_batches]).item())
        e2e_t.append(time.perf_counter() - t0)
    sync_all()
    e2e_ms = float(np.mean(e2e_t)) * 1e3
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    comm.all_reduce_max(t)
    e2e_ms = float(t.item())
    clk = clocks.stop() if clocks is not None else None
    tc_bwd = hot.work(B, T).tc["bwd"]
    tc_x3, tc_mode, cuda_graph = hot.tc_x3, hot.tc_mode, bool(
        hot.use_graphs and (world == 1 or hot.graph_collectives))
    fused = bool(getattr(hot, "ce_fused", False))
    del hot, resident, flush
    torch.cuda.empty_cache()

    # ---- the same workload through the reference-facing surface: RNNFullModel.fit_model on host id arrays (numpy in,
    #      History out); N = 1 only (the Keras surface drives one process)
    plugin = None
    if world == 1 and full:
        from seq_recommendations_b200.model import RNNFullModel
        from seq_recommendations_b200.optimizers import Adagrad
        # batches per timed epoch: enough that fit_model's per-call work (id conversion, range check, the one H2D copy of
        # the training set) is amortised as in a real epoch
        nb = 256 if step_ms < 2 else (32 if step_ms < 50 else 8)
        big_i, big_t = synthetic.make_batch(V, T, B * nb, seed=7)
        mdl = RNNFullModel(T, V, V, z_dim=H, rnn_type=cfg["cell"], z_to_z_activation=cfg["act"], y_to_y=False,
                           x_to_y=False, seed=0)
        mdl.compile_model(loss="categorical_crossentropy", metrics=[],
                          optimizer=Adagrad(lr=0.01, epsilon=1e-08, decay=0.0, clipnorm=1.))
        mdl.fit_model(big_i[:4 * B], big_t[:4 * B], n_epochs=1, batch_size=B, verbose=0)       # warm-up / graph capture
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hist = mdl.fit_model(big_i, big_t, n_epochs=1, batch_size=B, verbose=0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        plugin = {"value": B * nb / dt, "unit": "sequences/sec", "ms_per_step": dt / nb * 1e3,
                  "api": "RNNFullModel.fit_model(ids (N,T) int32 numpy, targets, n_epochs=1, batch_size=%d) -> History" % B,
                  "epoch_loss": float(hist.history["loss"][-1])}
        del mdl
        torch.cuda.empty_cache()

    if rank != 0:
        return None
    peaks = load_peaks()
    N = B * T * (world if vp else 1)                       # tokens one rank's logits kernels score per step
    work = algorithmic_work(cfg, N)
    if vp:                                                 # each rank scores all tokens against V / world items
        for k in ("ce_fwd_flops", "ce_bwd_flops"):
            work[k] /= world
    per_step = {k: v / steps for k, v in phases.items()}
    traffic, traffic_detail = load_traffic(name)
    # dominant phase: the logits kernels.  `fused` = forward statistics + dH from ONE logits pass (flash-style), then the
    # item-stationary dW kernel: 4 GEMM passes for 3 algorithmic GEMMs (x3: 12 bf16 passes); otherwise forward +
    # two recompute kernels: 5 GEMMs (x3: 15 passes)
    ce_ms = sum(v for k, v in per_step.items() if k.startswith("ce_fwd")) + per_step.get("ce_bwd", 0.0)
    ce_flops = work["ce_fwd_flops"] + work["ce_bwd_flops"]
    achieved = ce_flops / (ce_ms * 1e-3) / 1e12 if ce_ms > 0 else 0.0
    gemms_issued = (4 if fused else 5) * (3 if tc_x3 else 1) if tc_bwd else 5
    roofline = {
        "kernel": "logits path: seqrec_ce_%s (%s)" % (
            ("tc_* forward statistics + dH + dW_out", "tcgen05 bf16 %s, fp32 accumulate in TMEM" % (
                "3-pass hi/lo split" if tc_x3 else "single pass")) if tc_bwd else ("* SIMT", "fp32 SIMT")),
        "algorithmic_flops": ce_flops,
        "mma_flops_issued": work["ce_fwd_flops"] * gemms_issued,
        "issued_tflops": (work["ce_fwd_flops"] * gemms_issued / (ce_ms * 1e-3) / 1e12) if ce_ms > 0 else 0.0,
        "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
        "frac": achieved / peaks["bf16_sustained"], "traffic": traffic,
        "traffic_detail": traffic_detail,
        "peak_source": peaks["src"] + " bf16 sustained",
        "ms_per_launch": ce_ms,
        "others": hbm_evidence(name, work, per_step, peaks),
    }
    cpu = None
    if full and not args.no_cpu:
        # bounded sample: B scaled down until one oracle step costs about a second (factor stated in `sample`)
        sample_b = cpu_sample_batch(cfg, B)
        cpu = time_cpu(cfg, 8, 1 if sample_b < B else 2, budget_s=25.0, sample_b=sample_b)
    return {
        "value": world * B / (step_ms * 1e-3), "unit": "sequences/sec", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": step_ms,
        "dtype": {"x3": "f32 (bf16x3 split tensor-core GEMMs, fp32 accumulate; fp32 SIMT elsewhere)",
                  "bf16": "bf16 logits GEMMs, fp32 accumulate; fp32 elsewhere", "off": "f32"}[tc_mode],
        "config": config_dict(args, name, cfg, world, B, vp, cuda_graph),
        "clocks": clk,
        "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "sequences/sec", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": 2 * B * T * 4, "d2h_bytes_per_step": 4,
                "api": "HotPath.train_batch(pinned host ids, targets) -> loss.item()"},
        "e2e_plugin": plugin,
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "timed_steps")}
                         if cpu else None),
        "phases_ms": per_step,
        "scan": scan_info(cfg, B),
        "wall_s_timed_region": wall_s,
        "final_loss": final_loss,
    }


def hbm_evidence(name, work, per_step, peaks):
    """Gather / scatter-add against the HBM roofline.  The event-timed figure divides ALGORITHMIC bytes by the phase
    time: with Zipf-distributed ids the hot rows are served by the L2 and duplicates are merged in-warp, so it can
    exceed the HBM peak and is NOT an HBM fraction -- it is reported as `*_algorithmic_gbs`.  The HBM evidence proper is
    the committed ncu --set full capture of the two kernels (profiles/hbm_gather_scatter.json: dram bytes per launch
    and dram__throughput, at cfg4's 3 GB table and at cfg3 with uniform ids)."""
    out = {
        "gather_algorithmic_gbs": work["gather_bytes"] / (per_step.get("gather", 1e9) * 1e-3) / 1e9,
        "scatter_algorithmic_gbs": work["scatter_bytes"] / (per_step.get("scatter", 1e9) * 1e-3) / 1e9,
        "hbm_peak_gbs": peaks["hbm"],
        "note": "algorithmic bytes / event time; L2-served hot rows make this exceed DRAM traffic (see ncu)",
    }
    try:
        with open(os.path.join(ROOT, "profiles", "hbm_gather_scatter.json")) as f:
            out["ncu"] = json.load(f)
    except Exception:
        out["ncu"] = None
    try:
        # the history-feature kernel (datasets.build_xs on the device) is not part of a training step: its committed
        # probe (scripts/history_probe.py, CUDA events + ncu) rides along as evidence
        with open(os.path.join(ROOT, "profiles", "r2_history_features.json")) as f:
            h = json.load(f)
        out["history_features"] = {k: {"ms": v["ms"], "frac_of_hbm_peak": v["frac_of_hbm_peak"],
                                       "ncu_dram_throughput_pct": (v.get("ncu") or {}).get("dram_throughput_pct_of_peak")}
                                   for k, v in h["shapes"].items()}
    except Exception:
        out["history_features"] = None
    return out


def history_features_live(peaks, iters=5):
    """The history-feature kernel (seqrec_history_features: datasets.build_xs on the device, SURVEY 8(f) rank 1) timed
    live against the HBM roofline -- CUDA events on the launching stream, L2 flushed between launches; algorithmic
    bytes = n_seqs*T*V*4 written + the ragged corpus read once.  Not part of a training step: a side line of the run."""
    import ctypes
    import torch
    from seq_recommendations_b200._lib import call, ptr
    dev = torch.device("cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(0)
    out = {}
    for name, (n, T, V, lo, hi) in {"msnbc_like_V17_T50_200k_seqs": (200000, 50, 17, 2, 52),
                                     "cfg2_like_V10k_T50_512_seqs": (512, 50, 10000, 26, 52)}.items():
        lens = rng.integers(lo, hi, size=n)
        offs = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=offs[1:])
        items = torch.from_numpy(rng.integers(0, V, size=int(offs[-1])).astype(np.int32)).to(dev)
        d_offs = torch.from_numpy(offs).to(dev)
        table = torch.from_numpy(np.log(np.arange(hi + 1, dtype=np.float64) + 1.0).astype(np.float32)).to(dev)
        c = torch.empty((n, T, V), dtype=torch.float32, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        ms = []
        for i in range(3 + iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call("seqrec_history_features", ptr(items), ptr(d_offs), ptr(c), n, T, V, 1, ptr(table), hi + 1, ptr(err), st)
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ms.append(e0.elapsed_time(e1))
        alg = n * T * V * 4 + int(offs[-1]) * 4 + (n + 1) * 8
        t = float(np.median(ms))
        out[name] = {"ms": t, "algorithmic_bytes": alg, "achieved_gbs": alg / t / 1e6, "peak_gbs": peaks["hbm"],
                     "frac": alg / t / 1e6 / peaks["hbm"]}
        del items, d_offs, table, c
    del flush
    torch.cuda.empty_cache()
    return out


def parity_check(comm, rank, local):
    """N-rank step == rank-0 global-batch step (outside every timed region): relative error of the weights after three
    optimisation steps, data-parallel and vocabulary-parallel, so that the scaling record carries multi-GPU parity."""
    import torch
    from seq_recommendations_b200 import dist, synthetic
    from seq_recommendations_b200.engine import HotPath
    out = {}
    for key, (V, H, T, B, cell, vp) in (("dp", (900, 64, 10, 64, "GRU", False)),
                                        ("dp_rows", (60000, 64, 6, 64, "LSTM", False)),
                                        ("vp", (4096, 128, 8, 64, "GRU", True))):
        B = (B + comm.world - 1) // comm.world * comm.world
        act = "tanh" if cell == "GRU" else "relu"
        ws = synthetic.make_weights(cell, V, H, seed=3)
        steps = [synthetic.make_batch(V, T, B, seed=50 + s, min_len=1) for s in range(3)]
        hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc="x3", vocab_parallel=vp)
        # (lr = the reference's default, experiments_methods.py:21; the first Adagrad steps move every weight by ~lr, so
        # the weight error scales with it)
        hot.set_optimizer("adagrad", lr=0.01, epsilon=1e-8, clipnorm=1.0)
        lo, hi = dist.shard_rows(B, comm.rank, comm.world)
        losses = [float(hot.train_batch(i[lo:hi], t[lo:hi]).item()) for i, t in steps]
        mine = hot.get_weights()
        if rank == 0:
            solo = dist.Comm.__new__(dist.Comm)
            solo.enabled, solo.group, solo.rank, solo.world = False, None, 0, 1
            ref = HotPath(cell, act, V, H, V, weights=ws, comm=solo, tc="x3")
            ref.set_optimizer("adagrad", lr=0.01, epsilon=1e-8, clipnorm=1.0)
            ref_losses = [float(ref.train_batch(i, t).item()) for i, t in steps]
            errs = [float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30))
                    for a, b in zip(mine, ref.get_weights())]
            out[key] = max(errs)
            out[key + "_loss"] = max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses))
        comm.barrier()
    return out if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default=DEFAULT_CONFIG)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-table of the other BASELINE configurations")
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--tc", default="x3", choices=["x3", "bf16", "off"], help="logits GEMM mode (x3 = fp32-grade)")
    ap.add_argument("--vocab-parallel", type=int, default=-1,
                    help="1: column-shard W_out over the ranks (default for cfg4 when N > 1), 0: replicate")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline workload's last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    from seq_recommendations_b200 import synthetic
    cfg = dict(synthetic.CONFIGS[args.config])
    if args.impl == "reference":
        return run_reference(args, cfg, args.config)
    if args.config.startswith("cfg5"):
        print(json.dumps(run_scoring(args, cfg, args.config, dump=args.dump_outputs)))
        return

    import torch
    from seq_recommendations_b200 import dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))
    torch.cuda.set_device(local)
    comm = dist.init_from_env("nccl") if world > 1 else dist.Comm()

    head = measure_training(args, args.config, cfg, comm, rank, local, args.steps, args.warmup, full=True,
                            dump=args.dump_outputs)
    extra = {}
    if world > 1:
        # strong scaling of the same workload: the GLOBAL batch stays cfg B, every rank takes B / N sequences
        if cfg["B"] % world == 0:
            st = measure_training(args, args.config, cfg, comm, rank, local, args.steps, args.warmup, full=False,
                                  batch=cfg["B"] // world)
            if st is not None:
                extra["strong"] = {"global_batch": cfg["B"], "B_per_gpu": cfg["B"] // world, "value": st["value"],
                                   "unit": st["unit"], "ms_per_step": st["ms_per_step"], "e2e": st["e2e"]["value"],
                                   "scaling": "strong"}
        extra["parity_check"] = parity_check(comm, rank, local)
    if not args.no_sub:
        # the other BASELINE configurations, same measurement (weak scaling at N > 1), brief: value, ms/step, e2e,
        # roofline, clocks each
        sub = {}
        for name in ("cfg1_msnbc_lstm100", "cfg2_reddit_gru128", "cfg3_lstm256_50k"):
            if name == args.config:
                continue
            r = measure_training(args, name, dict(synthetic.CONFIGS[name]), comm, rank, local, args.steps, args.warmup,
                                 full=False)
            if r is not None:
                sub[name] = {k: r[k] for k in ("value", "unit", "ms_per_step", "config", "clocks", "phases_ms",
                                               "gpu_launches", "scan")}
                sub[name]["e2e"] = r["e2e"]["value"]
                sub[name]["roofline"] = {k: r["roofline"][k] for k in ("bound", "achieved", "peak", "unit", "frac",
                                                                      "ms_per_launch", "issued_tflops")}
        if world == 1:
            sc = run_scoring(args, dict(synthetic.CONFIGS["cfg5_score_gru256_100k"]), "cfg5_score_gru256_100k")
            sub["cfg5_score_gru256_100k"] = {k: sc[k] for k in ("metric", "value", "unit", "ms_per_step", "config",
                                                                 "clocks", "gpu_launches", "scan",
                                                                 "all_steps_target_prob")}
            sub["cfg5_score_gru256_100k"]["e2e"] = sc["e2e"]["value"]
            sub["cfg5_score_gru256_100k"]["roofline"] = {k: sc["roofline"][k] for k in ("bound", "achieved", "peak",
                                                                                         "unit", "frac")}
        extra["configs"] = sub
        if world == 1 and rank == 0:
            try:
                extra["history_features"] = history_features_live(load_peaks())
            except Exception as e:                 # a side line must never take the bench line down
                extra["history_features"] = {"error": repr(e)}
    if rank != 0:
        return
    line = {"metric": METRIC, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"}
    line.update(head)
    line.update(extra)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
