"""numpy mirror of record_enumerate_kernel's plan (csrc/records.cu): which grid window, level and noise window every slot
of an evaluation batch takes.  Pure integer arithmetic on uint64, so it must agree with the device bit for bit."""
from __future__ import annotations

import numpy as np

from tests.record_plan import mix64

_U = np.uint64


def n_items(R, T, W, stride, n_snr):
    return R * ((T - W) // stride + 1) * n_snr


def steps(R, T, W, stride, B, n_snr, world=1):
    """ceil(R * nper * n_snr / (world * B)): the batches that cover the set, the last one possibly ragged."""
    return -(-n_items(R, T, W, stride, n_snr) // (world * B))


def pair_noise(g, lvl, N, Tn, W, seed):
    """(noise record, noise offset) of (grid window g, level index lvl): a function of (seed, g, lvl) only."""
    with np.errstate(over="ignore"):
        hw = mix64(mix64(_U(seed & 0xFFFFFFFFFFFFFFFF) ^ mix64(np.asarray(g, dtype=np.uint64)))
                   ^ np.asarray(lvl, dtype=np.uint64))
        return mix64(hw + _U(1)) % _U(N), mix64(hw + _U(2)) % _U(Tn - W + 1)


def plan(R, T, N, Tn, W, stride, B, n_snr, seed, counter, rank=0, world=1):
    """(meta (B, 4) int64 = record, offset, noise record, noise offset; level index (B,) int64) of one rank's batch;
    slots past the end of the set have meta (-1, -1, -1, -1) and level -1."""
    nper = (T - W) // stride + 1
    e = np.arange(B, dtype=np.uint64) + _U(counter * world * B + rank * B)
    valid = e < _U(R * nper * n_snr)
    g, lvl = e // _U(n_snr), e % _U(n_snr)
    nrec, noff = pair_noise(g, lvl, N, Tn, W, seed)
    meta = np.stack([g // _U(nper), (g % _U(nper)) * _U(stride), nrec, noff], 1).astype(np.int64)
    lvl = lvl.astype(np.int64)
    meta[~valid] = -1
    lvl[~valid] = -1
    return meta, lvl
