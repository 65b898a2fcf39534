"""CPU checks of the record sampler (record_sampler.py, record_sample_kernel in csrc/records.cu): the index plan --
a keyed bijection per epoch, a new order every epoch, ranks partitioning the world batch -- through its numpy mirror
(tests/record_plan.py, which the GPU tests pin to the kernel bit for bit), the epoch length, and argument validation
that needs no device."""
import numpy as np
import pytest
import torch

from tests import record_plan as RP


@pytest.mark.parametrize("n", [1, 2, 3, 255, 256, 257, 4096, 48 * 2539])
def test_feistel_permutation_is_a_bijection(n):
    for key in (0, 12345, 2 ** 63 + 7):
        p = RP.feistel_perm(np.arange(n), n, RP.mix64(np.uint64(key)))
        assert p.dtype == np.uint64 and p.shape == (n,)
        assert np.array_equal(np.sort(p), np.arange(n, dtype=np.uint64)), (n, key)


def test_epochs_give_different_orders():
    R, T, W, B = 48, 2539 * 256, 256, 4096
    spe = RP.steps_per_epoch(R, T, W, W, B)
    assert spe == 29

    def epoch_items(e):
        return np.concatenate([RP.plan(R, T, 3, T, W, W, B, 5, 2023, e * spe + s)[0] for s in range(spe)])

    e0, e1 = epoch_items(0), epoch_items(1)
    for e in (e0, e1):       # every grid window at most once per epoch, all but the drop-last remainder
        key = e[:, 0] * T + e[:, 1]
        assert len(np.unique(key)) == spe * B
    assert not np.array_equal(e0[:, :2], e1[:, :2])
    # different orders, not just a shift: the first batch of the two epochs shares few windows
    first0 = set(map(tuple, e0[:B, :2])) & set(map(tuple, e1[:B, :2]))
    assert len(first0) < B // 4


def test_two_ranks_partition_the_world_batch():
    args = dict(R=5, T=10000, N=2, Tn=9000, W=256, stride=64, n_snr=5, seed=7)
    for ctr in (0, 1, 5, 300, 2 ** 31 - 1):
        m1, l1 = RP.plan(B=32, counter=ctr, **args)
        a, la = RP.plan(B=16, counter=ctr, rank=0, world=2, **args)
        b, lb = RP.plan(B=16, counter=ctr, rank=1, world=2, **args)
        assert np.array_equal(np.concatenate([a, b]), m1) and np.array_equal(np.concatenate([la, lb]), l1)


def test_plan_ranges_and_stride_one_crops():
    R, T, N, Tn, W = 3, 1000, 2, 700, 256
    for ctr in range(20):
        meta, lvl = RP.plan(R, T, N, Tn, W, 1, 64, 3, 11, ctr)
        assert (meta[:, 0] >= 0).all() and (meta[:, 0] < R).all()
        assert (meta[:, 1] >= 0).all() and (meta[:, 1] <= T - W).all()
        assert (meta[:, 2] >= 0).all() and (meta[:, 2] < N).all()
        assert (meta[:, 3] >= 0).all() and (meta[:, 3] <= Tn - W).all()
        assert (lvl >= 0).all() and (lvl < 3).all()
    meta = np.concatenate([RP.plan(R, T, N, Tn, W, 1, 64, 3, 11, c)[0] for c in range(RP.steps_per_epoch(
        R, T, W, 1, 64))])
    assert len(np.unique(meta[:, 0] * T + meta[:, 1])) == len(meta)      # crops without replacement


@pytest.mark.parametrize("R,T,W,stride,B,world", [(48, 650000, 256, 256, 256, 1), (48, 650000, 256, 256, 4096, 1),
                                                  (3, 1000, 256, 1, 64, 2), (1, 256, 256, 256, 1, 1),
                                                  (2, 5000, 512, 100, 7, 3), (1, 300, 256, 256, 2, 1)])
def test_steps_per_epoch_matches_the_formula(R, T, W, stride, B, world):
    from ecg_denoise_b200.record_sampler import steps_per_epoch
    assert steps_per_epoch(R, T, W, stride, B, world) == R * len(range(0, T - W + 1, stride)) // (world * B)
    assert steps_per_epoch(R, T, W, stride, B, world) == RP.steps_per_epoch(R, T, W, stride, B, world)


def test_bad_arguments_raise_without_a_device():
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.record_sampler import RecordSampler
    rec, nz = torch.zeros(2, 2, 1000), torch.zeros(1, 2, 800)
    bad = [
        dict(records=torch.zeros(2, 1000), noise=nz, batch=4),                     # not (R, leads, T)
        dict(records=torch.zeros(2, 13, 1000), noise=torch.zeros(1, 1, 800), batch=4),   # > 12 leads
        dict(records=rec, noise=torch.zeros(1, 3, 800), batch=4),                  # noise leads neither 1 nor 2
        dict(records=rec, noise=nz, batch=4, window=1001),                         # window > T
        dict(records=rec, noise=nz, batch=4, window=900),                          # window > Tn
        dict(records=rec, noise=nz, batch=0),
        dict(records=rec, noise=nz, batch=4, stride=0),
        dict(records=rec, noise=nz, batch=4, snr_db=()),
        dict(records=rec, noise=nz, batch=4, rank=2, world=2),
        dict(records=rec, noise=nz, batch=4, rank=-1, world=2),
        dict(records=rec, noise=nz, batch=7),                                      # 6 grid windows < one batch
        dict(records=rec, noise=nz, batch=4, world=2),                             # ... < world * batch
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            RecordSampler(**kw)
    with pytest.raises(_lib.RalenetError, match="cpu"):        # valid shapes, but the banks are not on a GPU
        RecordSampler(rec, nz, 4)
    with pytest.raises(_lib.RalenetError, match="cpu"):
        RecordSampler(rec, nz, 4, snr_db=-2.0, stride=1)
