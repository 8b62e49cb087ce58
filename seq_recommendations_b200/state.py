"""Carried recurrent state of a batch of sessions (inference only).

A state is h (n, H) float32 and, for LSTM models, the cell state c (n, H) float32; GRU and SimpleRNN models carry no c.
`HotPath.advance_state` continues the masked recurrence of the model from such a state over a chunk of new events and
returns the state after the chunk; the `*_from_state` scorers score the next item from it.  Row i is session i."""
import os

import numpy as np
import torch


def write_npz(filepath, arrays):
    """np.savez through a temp file and a rename: a reader never sees a torn archive."""
    d = os.path.dirname(filepath)
    if d and not os.path.exists(d):
        os.makedirs(d)
    tmp = "%s.tmp.%d" % (filepath, os.getpid())
    with open(tmp, "wb") as f:
        np.savez(f, **arrays)
    os.replace(tmp, filepath)


class RecurrentState(object):
    """h (n, H) float32, c (n, H) float32 for LSTM (None otherwise), the cell name and H."""

    def __init__(self, h, c, cell, H):
        self.h, self.c, self.cell, self.H = h, c, cell, int(H)
        if h.dim() != 2 or h.shape[1] != self.H or h.dtype != torch.float32:
            raise ValueError("h must be (n, %d) float32, got %s %s" % (self.H, tuple(h.shape), h.dtype))
        if (cell == "LSTM") != (c is not None):
            raise ValueError("an LSTM state carries c; a %s state does not" % cell)
        if c is not None and (c.shape != h.shape or c.dtype != torch.float32 or c.device != h.device):
            raise ValueError("c must match h: (n, %d) float32 on %s" % (self.H, h.device))

    def __len__(self):
        return self.h.shape[0]

    @classmethod
    def zeros(cls, n, cell, H, device):
        z = lambda: torch.zeros((int(n), int(H)), dtype=torch.float32, device=device)
        return cls(z(), z() if cell == "LSTM" else None, cell, H)

    def check(self, cell, H, n=None):
        """ValueError unless this state belongs to a (cell, H) model (and has n rows, when n is given)."""
        if self.cell != cell or self.H != int(H):
            raise ValueError("state of a %s-%d model used with a %s-%d model" % (self.cell, self.H, cell, int(H)))
        if n is not None and len(self) != int(n):
            raise ValueError("state holds %d sessions, the batch %d" % (len(self), int(n)))

    def _index(self, index):
        if isinstance(index, slice):
            return index
        return torch.as_tensor(np.asarray(index) if not isinstance(index, torch.Tensor) else index,
                               device=self.h.device).long()

    def take(self, index):
        """The states of a subset of sessions (a copy)."""
        i = self._index(index)
        return RecurrentState(self.h[i].clone(), None if self.c is None else self.c[i].clone(), self.cell, self.H)

    def put(self, index, other):
        """Writes the rows of `other` back into the sessions `index`, in place."""
        other.check(self.cell, self.H)
        i = self._index(index)
        n = len(range(*i.indices(len(self)))) if isinstance(i, slice) else i.numel()
        if n != len(other):
            raise ValueError("%d rows to put, %d indices" % (len(other), n))
        self.h[i] = other.h.to(self.h.device)
        if self.c is not None:
            self.c[i] = other.c.to(self.c.device)

    def to(self, device):
        return RecurrentState(self.h.to(device), None if self.c is None else self.c.to(device), self.cell, self.H)

    def save(self, path):
        arrays = dict(h=self.h.cpu().numpy(), cell=np.asarray(self.cell), H=np.asarray(self.H))
        if self.c is not None:
            arrays["c"] = self.c.cpu().numpy()
        write_npz(path, arrays)

    @classmethod
    def load(cls, path, device="cpu"):
        with np.load(path) as z:
            c = torch.from_numpy(z["c"]).to(device) if "c" in z.files else None
            return cls(torch.from_numpy(z["h"]).to(device), c, str(z["cell"]), int(z["H"]))
