"""ctypes binding of the C-ABI in include/seqrec_b200.h (libseqrec_b200.so, built in-tree by build.py).

There is NO fallback: if the shared library is missing or a call fails, this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libseqrec_b200.so")

CELL = {"simpleRNN": 0, "LSTM": 1, "GRU": 2}
ACT = {"relu": 0, "tanh": 1, "linear": 2}

_p = ctypes.c_void_p
_i = ctypes.c_int
_l = ctypes.c_int64
_f = ctypes.c_float
_u64 = ctypes.c_uint64

# name -> argtypes; must list every symbol include/seqrec_b200.h declares (tests/test_abi.py checks this)
SIGNATURES = {
    "seqrec_device_cc": [],
    "seqrec_abi_version": [],
    "seqrec_launch_count": [_i],
    "seqrec_pad_sequences": [_p, _p, _p, _p, _l, _i, _p],
    "seqrec_history_features": [_p, _p, _p, _l, _i, _i, _i, _p, _i, _p, _p],
    "seqrec_format_batch": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p],
    "seqrec_gather_rows": [_p, _p, _p, _p, _p, _p, _l, _i, _i, _p],
    "seqrec_scatter_add_rows": [_p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _p],
    "seqrec_mark_rows": [_p, _p, _p, _p, _p, _l, _i, _p],
    "seqrec_gemm_nn": [_p, _p, _p, _p, _i, _i, _i, _i, _p],
    "seqrec_gemm_tc": [_p, _p, _p, _p, _p, _p, _l, _i, _i, _l, _l, _l, _i, _i, _p],
    "seqrec_gemm_tn_atomic": [_p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_forward": [_i, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_forward_state": [_i, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_backward": [_i, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_forward_rd": [_i, _i, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_backward_rd": [_i, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_weight_grad_rd": [_i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_needs_ut": [_i, _i],
    "seqrec_rnn_tc_applicable": [_i, _i],
    "seqrec_rnn_tc_max_clusters": [_i, _i],
    "seqrec_rnn_tc_forward": [_i, _i, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_tc_forward_state": [_i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_tc_backward": [_i, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_tc_debug_buffer": [_p],
    "seqrec_rnn_weight_grad": [_i, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rnn_weight_grad_tc": [_i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_transpose": [_p, _p, _i, _i, _p],
    "seqrec_ce_forward": [_p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _p],
    "seqrec_ce_finalize": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _p],
    "seqrec_ce_finalize_mean": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _p, _p],
    "seqrec_ce_backward": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _i, _p],
    "seqrec_ce_tc_forward": [_p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _i, _i, _i, _p],
    "seqrec_ce_tc_forward_rank": [_p] * 9 + [_i, _p, _l, _i, _i, _i, _i, _i, _p],
    "seqrec_target_rank": [_p, _p, _p, _p, _p, _i, _p, _l, _i, _i, _i, _i, _i, _p],
    "seqrec_ce_tc_partials": [_l, _i, _i],
    "seqrec_ce_tc_backward": [_p] * 16 + [_l, _i, _i, _i, _i, _l, _i, _i, _i, _i, _i, _p, _p, _p, _p],
    "seqrec_ce_tc_fused": [_p] * 11 + [_l, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "seqrec_ce_dh_finish": [_p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _p, _p, _p],
    "seqrec_compact_tokens": [_p, _p, _l, _p, _p, _p, _p, _p],
    "seqrec_split_bf16_both_rows": [_p, _p, _p, _p, _p, _p, _p, _p, _l, _l, _l, _l, _p],
    "seqrec_target_logit": [_p, _p, _p, _p, _p, _p, _l, _i, _i, _p, _p, _p],
    "seqrec_predict_probs": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p],
    "seqrec_topk": [_p, _p, _p, _p, _p, _p, _p, _l, _i, _i, _i, _p],
    "seqrec_topk_tc": [_p] * 11 + [_l, _i, _i, _i, _i, _p],
    "seqrec_topk_merge": [_p, _p, _i, _l, _p, _p, _l, _i, _p],
    "seqrec_candidate_logits": [_p, _p, _p, _p, _l, _p, _l, _i, _i, _i, _i, _p],
    "seqrec_candidate_order": [_p, _p, _i, _l, _p, _p, _i, _p, _p, _p, _p, _p, _p],
    "seqrec_sample_items": [_p, _i, _p, _p, _i, _u64, _p, _p],
    "seqrec_gather_columns": [_p, _l, _p, _p, _p, _i, _i, _p, _p, _p],
    "seqrec_sampled_softmax_rows": [_p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p],
    "seqrec_target_columns": [_p, _p, _p, _l, _p, _p, _p, _p, _p, _l, _i, _p],
    "seqrec_scatter_add_columns": [_p, _p, _p, _i, _i, _p, _l, _p, _p],
    "seqrec_add_rows": [_p, _p, _p, _p, _l, _i, _p],
    "seqrec_softmax_rows_stats": [_p, _p, _p, _p, _p, _l, _i, _p],
    "seqrec_softmax_rows_dlogit": [_p, _p, _p, _p, _p, _l, _i, _p],
    "seqrec_softmax_rows_probs": [_p, _p, _p, _p, _i, _i, _i, _p],
    "seqrec_rows_rank": [_p, _p, _p, _l, _i, _p],
    "seqrec_gemm_nt": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "seqrec_colsum": [_p, _p, _l, _i, _i, _p],
    "seqrec_diag_constraint": [_p, _i, _i, _p],
    "seqrec_likelihood": [_p, _p, _l, _i, _i, _p, _p],
    "seqrec_likelihood_cut": [_p, _p, _l, _i, _i, ctypes.c_double, _p, _p],
    "seqrec_rank_metrics": [_p, _l, _p, _i, _p, _p],
    "seqrec_sumsq": [_p, _l, _p, _p],
    "seqrec_sumsq_rows": [_p, _p, _p, _i, _i, _p, _p],
    "seqrec_adagrad": [_p, _p, _p, _l, _f, _f, _f, _p, _p, _p],
    "seqrec_adagrad_rows": [_p, _p, _p, _p, _p, _p, _i, _i, _f, _f, _f, _p, _p, _p],
    "seqrec_adam": [_p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _f, _p, _p, _p, _p],
    "seqrec_adam_table": [_p, _p, _p, _p, _p, _l, _i, _f, _f, _f, _f, _f, _f, _p, _p, _p, _p],
    "seqrec_dropout_mask": [_p, _l, _f, _u64, _u64, _p],
    "seqrec_dropout_mask_dev": [_p, _l, _f, _u64, _p, _p],
    "seqrec_split_bf16": [_p, _p, _p, _p, _l, _l, _l, _i, _p],
    "seqrec_split_bf16_colsum": [_p, _p, _p, _p, _l, _i, _p],
    "seqrec_split_bf16_both": [_p, _p, _p, _p, _p, _p, _l, _l, _l, _l, _p],
}

_lib = None


class SeqrecError(RuntimeError):
    pass


def load():
    """Load libseqrec_b200.so; raise loudly when it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SeqrecError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  seq_recommendations_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the .so is stale
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    _lib = lib
    return lib


def call(name, *args):
    """Invoke one C-ABI entry point; non-zero status raises SeqrecError."""
    fn = getattr(load(), name)
    rc = fn(*args)
    if rc != 0:
        raise SeqrecError("%s failed with status %d" % (name, rc))
    return rc


def launch_count(reset=False):
    """Kernels launched by the library so far (bench.py's gpu_launches)."""
    return load().seqrec_launch_count(1 if reset else 0)


def ptr(t):
    """Device pointer of a torch tensor (or NULL for None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())
