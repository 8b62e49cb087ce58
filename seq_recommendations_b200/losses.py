"""Training objectives beyond the reference's `categorical_crossentropy`, and the host half of their setup.

`SampledSoftmax(num_sampled, weights=None)` trains on a sampled softmax with log-Q correction instead of the full-catalog
softmax: every step draws `num_sampled` item ids S with replacement from q (uniform, or weights / sum(weights)) and
scores each token against its target and those S shared items,

    l_0 = o_y - log Q(y),   l_j = o_{s_j} - log Q(s_j)  (dropped where s_j == y),   loss = -l_0 + log sum_j exp(l_j)

with o = h . W_out + b_out and log Q(v) = log(S q(v)) -- TF `sampled_softmax_loss` with `subtract_log_q` and
`remove_accidental_hits`, without Keras' 1e-7 probability clip.  A step then costs S columns instead of V.  Only the
training loss changes: `val_loss`, `evaluate` and the ranking metrics stay full-softmax.

    model.compile_model(loss=losses.SampledSoftmax(8192, weights=counts ** 0.75), optimizer=Adagrad(lr=0.05))

The draw runs on the device (csrc/sampled.cu); the Vose alias table and the log Q table it reads are built here, once,
in float64."""
import numpy as np

# include/seqrec_b200.h SEQREC_MAX_SAMPLED: the rows kernel keeps the S sampled ids in shared memory to find the
# accidental hits, 128 KB at this bound
MAX_SAMPLED = 32768


class SampledSoftmax(object):
    """Loss spec for `compile_model(loss=...)`: num_sampled draws per step from q = uniform (weights None) or
    weights / sum(weights) (V finite positive values, e.g. item counts ** 0.75)."""
    kind = "sampled_softmax"

    def __init__(self, num_sampled, weights=None):
        self.num_sampled = _check_num_sampled(num_sampled)
        self.weights = None if weights is None else _check_weights(weights)

    def __repr__(self):
        return "SampledSoftmax(num_sampled=%d%s)" % (self.num_sampled, "" if self.weights is None else ", weights=...")


def _check_num_sampled(num_sampled):
    if isinstance(num_sampled, (bool, np.bool_)) or not isinstance(num_sampled, (int, np.integer)):
        raise ValueError("num_sampled must be an integer, got %r" % (num_sampled,))
    if not 1 <= int(num_sampled) <= MAX_SAMPLED:
        raise ValueError("num_sampled must be in [1, %d], got %d" % (MAX_SAMPLED, int(num_sampled)))
    return int(num_sampled)


def _check_weights(weights):
    w = np.asarray(weights, dtype=np.float64)
    if w.ndim != 1 or w.size == 0:
        raise ValueError("weights must be a 1-D array of one value per item, got shape %s" % (w.shape,))
    if not np.all(np.isfinite(w)) or not np.all(w > 0):
        raise ValueError("weights must be finite and > 0 for every item (log Q of a zero-weight target is infinite)")
    return w


def check_sampled(num_sampled, weights, V):
    """Validated (S, q) for a catalog of V items: 1 <= S <= min(V, MAX_SAMPLED); q float64 (V,), or None = uniform."""
    S = _check_num_sampled(num_sampled)
    if S > V:
        raise ValueError("num_sampled (%d) must not exceed the catalog size (%d)" % (S, V))
    if weights is None:
        return S, None
    w = _check_weights(weights)
    if w.shape != (V,):
        raise ValueError("weights must have shape (%d,), got %s" % (V, w.shape))
    return S, w / w.sum()


def alias_table(q):
    """Vose's alias table of q (float64, sums to 1): column c of V is kept with probability thr[c] / 2^32 and gives way
    to alias[c] otherwise.  Returns (thr uint32, alias int32).  A full column keeps itself (alias = c)."""
    V = q.shape[0]
    p = np.asarray(q, dtype=np.float64) * V
    thr = np.ones(V, dtype=np.float64)
    alias = np.arange(V, dtype=np.int64)
    small = [int(i) for i in np.nonzero(p < 1.0)[0]]
    large = [int(i) for i in np.nonzero(p >= 1.0)[0]]
    while small and large:
        s, l = small.pop(), large.pop()
        thr[s] = p[s]
        alias[s] = l
        p[l] = (p[l] + p[s]) - 1.0
        (small if p[l] < 1.0 else large).append(l)
    # what is left is full up to rounding: thr stays 1, alias stays the column itself
    t = np.minimum(np.rint(thr * 4294967296.0), 4294967295.0)
    return t.astype(np.uint32), alias.astype(np.int32)


def log_q(S, q, V):
    """log(S q(v)) as float32 (V,), computed in float64: the expected count of v among the S draws."""
    if q is None:
        return np.full(V, np.log(S / V), dtype=np.float32)
    return np.log(S * q).astype(np.float32)
