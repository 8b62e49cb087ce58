"""Optimizer spec objects with the constructor surface of `keras.optimizers` as the reference uses it
(experiments_methods.py:10, :41: `Adagrad(lr=lr, epsilon=1e-08, decay=0.0, clipnorm=1.)`).  They only carry
hyper-parameters; the arithmetic is the K8 kernels (csrc/optim.cu)."""


class Optimizer(object):
    kind = None

    def __init__(self, clipnorm=None, clipvalue=None):
        if clipvalue is not None:
            raise NotImplementedError("clipvalue is never used by the reference")
        self.clipnorm = clipnorm


class Adagrad(Optimizer):
    kind = "adagrad"

    def __init__(self, lr=0.01, epsilon=1e-8, decay=0.0, **kwargs):
        Optimizer.__init__(self, **kwargs)
        self.lr = lr
        self.epsilon = epsilon
        self.decay = decay


class Adam(Optimizer):
    """Keras 2.0.x Adam: the update is dense -- every coordinate moves at every step, rows of the input table that a
    batch does not touch included (their gradient is zero; m and v decay)."""
    kind = "adam"

    def __init__(self, lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-8, decay=0.0, **kwargs):
        Optimizer.__init__(self, **kwargs)
        self.lr = lr
        self.beta_1 = beta_1
        self.beta_2 = beta_2
        self.epsilon = epsilon
        self.decay = decay


def kind_of(optimizer):
    return getattr(optimizer, "kind", type(optimizer).__name__.lower())


def resolve(optimizer):
    """Accept an optimizer object (anything exposing lr / epsilon / decay / clipnorm, e.g. a Keras Adagrad, and for
    Adam beta_1 / beta_2) or the name 'adagrad'.  `compile_model`'s default string 'adam' (model.py:176) is accepted at
    compile time but the reference never trains with it; fitting with it raises -- train with an `Adam(...)` object."""
    if isinstance(optimizer, str):
        if optimizer.lower() == "adagrad":
            return Adagrad()
        return optimizer.lower()
    kind = kind_of(optimizer)
    if kind not in ("adagrad", "adam"):
        return kind
    return optimizer
