"""numpy mirror of record_sample_kernel's index plan (csrc/records.cu): which clean window, noise window and SNR level
every slot of a batch draws.  Pure integer arithmetic on uint64, so it must agree with the device bit for bit."""
from __future__ import annotations

import numpy as np

_U = np.uint64
ROUNDS = 4


def mix64(z):
    """SplitMix64 finaliser (common.cuh), elementwise on uint64 with wrap-around."""
    with np.errstate(over="ignore"):
        z = np.asarray(z, dtype=np.uint64) + _U(0x9e3779b97f4a7c15)
        z = (z ^ (z >> _U(30))) * _U(0xbf58476d1ce4e5b9)
        z = (z ^ (z >> _U(27))) * _U(0x94d049bb133111eb)
        return z ^ (z >> _U(31))


def feistel_perm(x, n: int, key) -> np.ndarray:
    """keyed bijection of [0, n): balanced Feistel network on 2h bits, cycle walking back into [0, n)."""
    h = 1
    while (1 << (2 * h)) < n:
        h += 1
    m = _U((1 << h) - 1)
    with np.errstate(over="ignore"):
        rks = [mix64(_U(key) + _U(k)) for k in range(ROUNDS)]
    x = np.array(x, dtype=np.uint64, ndmin=1)
    todo = np.ones(x.shape, dtype=bool)
    while todo.any():
        l, r = x[todo] >> _U(h), x[todo] & m
        for rk in rks:
            l, r = r, l ^ (mix64(r ^ rk) & m)
        x[todo] = (l << _U(h)) | r
        todo = x >= _U(n)
    return x


def steps_per_epoch(R, T, W, stride, B, world=1):
    return R * ((T - W) // stride + 1) // (world * B)


def plan(R, T, N, Tn, W, stride, B, n_snr, seed, counter, rank=0, world=1):
    """(meta (B, 4) int64 = record, offset, noise record, noise offset; level index (B,)) of one rank's batch."""
    nper = (T - W) // stride + 1
    n = R * nper
    spe = n // (world * B)
    assert spe > 0
    ctr = counter & 0xFFFFFFFF
    epoch, step = ctr // spe, ctr % spe
    seed = _U(seed & 0xFFFFFFFFFFFFFFFF)
    slot = np.arange(B, dtype=np.uint64) + _U(rank * B)
    g = _U(step * world * B) + slot
    with np.errstate(over="ignore"):
        item = feistel_perm(g, n, mix64(seed ^ mix64(_U(2 * epoch))))
        hw = mix64(mix64(seed ^ mix64(_U(2 * ctr + 1))) ^ slot)
        nrec = mix64(hw + _U(1)) % _U(N)
        noff = mix64(hw + _U(2)) % _U(Tn - W + 1)
        lvl = mix64(hw + _U(3)) % _U(n_snr)
    meta = np.stack([item // _U(nper), (item % _U(nper)) * _U(stride), nrec, noff], 1).astype(np.int64)
    return meta, lvl.astype(np.int64)
