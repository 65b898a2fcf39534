"""CPU checks of the held-out evaluator (evaluate.py, record_enumerate_kernel in csrc/records.cu): the ordered plan
through its numpy mirror (tests/eval_plan.py, which the GPU tests pin to the kernel bit for bit) -- every (grid window,
level) pair once over all batches and ranks, the ragged tail, a noise pairing that does not depend on the batch or the
rank split -- and argument validation that needs no device."""
import numpy as np
import pytest
import torch

from tests import eval_plan as EP

SHAPES = [  # R, T, N, Tn, W, stride, B, n_snr, world
    (3, 1000, 2, 700, 256, 256, 4, 5, 1),
    (3, 1000, 2, 700, 256, 100, 7, 3, 2),
    (5, 3000, 3, 2500, 256, 64, 16, 5, 3),
    (1, 256, 1, 256, 256, 256, 1, 1, 1),
    (2, 5000, 2, 5000, 512, 1, 64, 2, 4),
    (4, 2600, 3, 2600, 256, 256, 9, 5, 2),
]


def _all_slots(R, T, N, Tn, W, stride, B, n_snr, world, seed=7):
    """(meta, level) of every slot in global slot order k * world * B + r * B + i."""
    metas, lvls = [], []
    for k in range(EP.steps(R, T, W, stride, B, n_snr, world)):
        for r in range(world):
            m, l = EP.plan(R, T, N, Tn, W, stride, B, n_snr, seed, k, rank=r, world=world)
            metas.append(m)
            lvls.append(l)
    return np.concatenate(metas), np.concatenate(lvls)


@pytest.mark.parametrize("R,T,N,Tn,W,stride,B,n_snr,world", SHAPES)
def test_every_pair_once_and_the_tail_is_the_last_slots(R, T, N, Tn, W, stride, B, n_snr, world):
    meta, lvl = _all_slots(R, T, N, Tn, W, stride, B, n_snr, world)
    nper = (T - W) // stride + 1
    n = EP.n_items(R, T, W, stride, n_snr)
    steps = EP.steps(R, T, W, stride, B, n_snr, world)
    assert steps == -(-R * len(range(0, T - W + 1, stride)) * n_snr // (world * B))
    valid = lvl >= 0
    assert valid.sum() == n
    tail = steps * world * B - n
    assert 0 <= tail < world * B
    assert valid[:n].all() and not valid[n:].any()            # the invalid slots are exactly the last ones
    assert (meta[~valid] == -1).all()
    g = meta[valid, 0] * nper + meta[valid, 1] // stride
    assert (meta[valid, 1] % stride == 0).all()
    pairs = g * n_snr + lvl[valid]
    assert np.array_equal(pairs, np.arange(n))                # every (grid window, level) once, in order
    assert (meta[valid, 2] >= 0).all() and (meta[valid, 2] < N).all()
    assert (meta[valid, 3] >= 0).all() and (meta[valid, 3] <= Tn - W).all()


def test_noise_pick_does_not_depend_on_batch_world_or_rank():
    R, T, N, Tn, W, stride, n_snr, seed = 4, 3000, 3, 2000, 256, 128, 5, 11
    ref = None
    for B, world in ((1, 1), (7, 1), (16, 2), (5, 3), (64, 4)):
        meta, lvl = _all_slots(R, T, N, Tn, W, stride, B, n_snr, world, seed)
        v = lvl >= 0
        got = {(int(m[0]), int(m[1]), int(l)): (int(m[2]), int(m[3])) for m, l in zip(meta[v], lvl[v])}
        if ref is None:
            ref = got
        assert got == ref, (B, world)
    # ... and pairs differ across levels and seeds (the pick is keyed by both)
    m5, l5 = EP.plan(R, T, N, Tn, W, stride, 200, n_snr, seed, 0)
    assert len({(int(a), int(b)) for a, b in m5[:, 2:]}) > 100
    m6, _ = EP.plan(R, T, N, Tn, W, stride, 200, n_snr, seed + 1, 0)
    assert not np.array_equal(m5[:, 2:], m6[:, 2:])


def test_steps_attribute_matches_the_mirror_without_a_device():
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.evaluate import RecordEvaluator
    rec, nz = torch.zeros(3, 2, 1000), torch.zeros(2, 1, 700)
    # on the CPU the constructor gets as far as the placement check, after the grid size is known
    with pytest.raises(_lib.RalenetError, match="cpu"):
        RecordEvaluator(rec, nz, 7, stride=100, snr_db=(-1, 0, 1))
    for (B, stride, levels, world) in ((7, 100, (-1, 0, 1), 2), (4, 256, (0,), 1), (1000, 1, (-4, 4), 3)):
        ev = RecordEvaluator.__new__(RecordEvaluator)
        ev._check_grid(3, (1000 - 256) // stride + 1, [float(v) for v in levels], B, world)
        assert ev.steps == EP.steps(3, 1000, 256, stride, B, len(levels), world)
        assert ev.n_items == EP.n_items(3, 1000, 256, stride, len(levels))


def test_bad_arguments_raise_without_a_device():
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.evaluate import RecordEvaluator
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
        dict(records=rec, noise=nz, batch=4, snr_db=(0, 2, 0)),                    # a level twice
        dict(records=rec, noise=nz, batch=4, rank=2, world=2),
        dict(records=rec, noise=nz, batch=4, rank=-1, world=2),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            RecordEvaluator(**kw)
    # a batch larger than the whole set is fine for evaluation (one ragged step); only the placement fails here
    for kw in (dict(batch=10 ** 5), dict(batch=4, world=8, rank=7), dict(batch=4, snr_db=-2.0, stride=1)):
        with pytest.raises(_lib.RalenetError, match="cpu"):
            RecordEvaluator(rec, nz, **kw)
