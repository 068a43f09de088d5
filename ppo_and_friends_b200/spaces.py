"""
Minimal Box / Discrete / MultiDiscrete / MultiBinary stand-ins with the attributes the update path reads from gymnasium
spaces (`shape`, `dtype`, `low`, `high`, `n`, `nvec`, `start`).  gymnasium is not part of this image; real gymnasium
spaces work unchanged because the policy only duck-types these attributes.
"""
import numpy as np


class Box:
    def __init__(self, low, high, shape=None, dtype=np.float32):
        shape = np.shape(low) if shape is None else tuple(shape)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype=self.dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=self.dtype), self.shape).copy()


class Discrete:
    def __init__(self, n, start=0):
        self.n = int(n)
        self.start = start
        self.shape = ()
        self.dtype = np.dtype(np.int64)


class MultiDiscrete:
    def __init__(self, nvec, start=None):
        self.nvec = np.asarray(nvec, dtype=np.int64)
        self.start = None if start is None else np.asarray(start, dtype=np.int64)
        self.shape = self.nvec.shape
        self.dtype = np.dtype(np.int64)


class MultiBinary:
    """`n` binary actions; like gymnasium, `n` may also be a shape (which the policy refuses unless it is 1-D)."""

    def __init__(self, n):
        self.n = n
        self.shape = tuple(int(d) for d in np.atleast_1d(n))
        self.dtype = np.dtype(np.int8)
