"""GPU checks of the device-resident record sampler (record_sampler.py, record_sample_kernel in csrc/records.cu):
the drawn plan against its numpy mirror bit for bit, the clean windows against the oracle's record cut, the noisy
windows against the oracle's SNR mix, epoch coverage, rank slices, and both trainers' step_synth."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ralenet_oracle as O
from oracle import synth_weights as SW
from tests import record_plan as RP
from tests.common import rel_rms_err

pytestmark = pytest.mark.gpu
LEVELS = (-4.0, -2.0, 0.0, 2.0, 4.0)


def _banks(leads, noise_leads, R=4, T=3000, N=3, Tn=2500, seed=0):
    rs = np.random.RandomState(seed + leads)
    rec = rs.standard_normal((R, leads, T)).astype(np.float32) * 2 + 0.7
    nz = rs.standard_normal((N, noise_leads, Tn)).astype(np.float32) * 0.5
    return torch.from_numpy(rec).cuda(), torch.from_numpy(nz).cuda()


def _sampler(rec, nz, B, **kw):
    from ecg_denoise_b200.record_sampler import RecordSampler
    return RecordSampler(rec, nz, B, **kw)


CASES = [(2, 2, 256), (2, 1, 1), (12, 1, 256), (12, 12, 1)]       # (leads, noise leads, stride)


@pytest.mark.parametrize("leads,noise_leads,stride", CASES)
def test_plan_matches_numpy_mirror_and_windows_match_the_oracle(leads, noise_leads, stride):
    rec, nz = _banks(leads, noise_leads)
    R, _, T = rec.shape
    N, _, Tn = nz.shape
    W, B, seed = 256, 16, 99
    sp = _sampler(rec, nz, B, window=W, stride=stride, snr_db=LEVELS, seed=seed)
    assert (sp.B, sp.leads, sp.L) == (B, leads, W)
    assert sp.steps_per_epoch == RP.steps_per_epoch(R, T, W, stride, B)
    win_ref, _ = O.records_to_windows(rec.double().cpu(), W, stride)
    nper = (T - W) // stride + 1
    levels = torch.tensor(LEVELS, dtype=torch.float32)
    spe = sp.steps_per_epoch
    for ctr in (0, 1, 2, spe - 1, spe, spe + 3, 5 * spe + 1, 2 ** 31 - 1):
        noisy, clean = sp.batch(counter=torch.tensor([ctr], dtype=torch.int32, device="cuda"))
        meta, snr = sp.meta.cpu().numpy(), sp.snr.cpu()
        meta_ref, lvl_ref = RP.plan(R, T, N, Tn, W, stride, B, len(LEVELS), seed, ctr)
        assert np.array_equal(meta.astype(np.int64), meta_ref), ctr
        assert torch.equal(snr, levels[torch.from_numpy(lvl_ref)]), ctr
        idx = torch.from_numpy(meta_ref[:, 0] * nper + meta_ref[:, 1] // stride)
        ref = win_ref[idx].numpy()
        assert rel_rms_err(clean.double().cpu().numpy(), ref) <= 1e-6, ctr
        nref = torch.stack([nz[m[2], :, m[3]:m[3] + W].cpu() for m in meta_ref])
        nref = nref[:, [l % noise_leads for l in range(leads)]]
        assert torch.equal(sp.noise.cpu(), nref), ctr
        mix_ref = O.snr_mix(clean.double().cpu(), nref.double(), snr.double())
        assert rel_rms_err(noisy.double().cpu().numpy(), mix_ref.numpy()) <= 1e-5, ctr
        n = (noisy.double() - clean.double()).reshape(B, -1)
        realised = 10 * torch.log10((clean.double().reshape(B, -1) ** 2).mean(1) / (n ** 2).mean(1))
        assert float((realised.cpu() - snr.double()).abs().max()) < 0.01, ctr
    noisy0, _ = sp.batch(counter=0)
    noisy0b, _ = sp.batch()                    # None = counter 0
    assert torch.equal(noisy0, noisy0b)


def test_no_znorm_and_single_level():
    rec, nz = _banks(2, 2)
    sp = _sampler(rec, nz, 8, znorm=False, snr_db=3.0, seed=5)
    noisy, clean = sp.batch(counter=4)
    meta = sp.meta.cpu().numpy()
    ref = torch.stack([rec[m[0], :, m[1]:m[1] + 256].cpu() for m in meta])
    assert torch.equal(clean.cpu(), ref) and bool((sp.snr == 3.0).all())


@pytest.mark.parametrize("stride", [256, 1])
def test_one_epoch_visits_every_grid_window_once(stride):
    rec, nz = _banks(2, 1, R=3, T=256 * 40 + 17)
    R, _, T = rec.shape
    B = 8 if stride == 256 else 512
    sp = _sampler(rec, nz, B, stride=stride, seed=3)
    nper = (T - 256) // stride + 1
    spe = sp.steps_per_epoch
    assert spe == R * nper // B
    ctr = torch.zeros(1, dtype=torch.int32, device="cuda")
    for epoch in range(2):
        seen = []
        for _ in range(spe):
            sp.batch(ctr)
            seen.append(sp.meta.clone())
            ctr += 1
        m = torch.cat(seen).cpu()
        assert bool((m[:, 1] % stride == 0).all()) and bool((m[:, 1] <= T - 256).all())
        key = m[:, 0] * nper + m[:, 1] // stride
        assert len(torch.unique(key)) == spe * B                   # each grid window at most once
        assert R * nper - spe * B < B                              # all of them up to the drop-last remainder
        if epoch == 0:
            first = key
    assert not torch.equal(first, key)                             # a new order in the next epoch


def test_two_ranks_concatenate_to_the_world_batch():
    rec, nz = _banks(2, 2)
    B = 16
    s1 = _sampler(rec, nz, 2 * B, stride=64, seed=21, rank=0, world=1)
    s_a = _sampler(rec, nz, B, stride=64, seed=21, rank=0, world=2)
    s_b = _sampler(rec, nz, B, stride=64, seed=21, rank=1, world=2)
    assert s_a.steps_per_epoch == s_b.steps_per_epoch == s1.steps_per_epoch
    for ctr in (0, 3, s1.steps_per_epoch + 1):
        full = s1.batch(ctr) + (s1.meta.clone(), s1.snr.clone())
        a = s_a.batch(ctr) + (s_a.meta.clone(), s_a.snr.clone())
        b = s_b.batch(ctr) + (s_b.meta.clone(), s_b.snr.clone())
        for u, v, w in zip(full, a, b):
            assert torch.equal(u, torch.cat([v, w])), ctr


def _ralenet(seed=2023):
    from ecg_denoise_b200.model import transformer
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(SW.make_state_dict("rw", 1, seed), strict=True)
    return m.cuda().train()


def test_fused_trainer_graphed_step_synth_is_bit_identical_to_eager_steps():
    from ecg_denoise_b200.engine import FusedTrainer
    rec, nz = _banks(2, 1, R=4, T=20000)
    sp = _sampler(rec, nz, 64, seed=8)
    ma, mb = _ralenet(), _ralenet()
    ta = FusedTrainer(ma, use_graph=True, deterministic=True)
    tb = FusedTrainer(mb, use_graph=False, deterministic=True)
    la = [ta.step_synth(sp)[0].clone() for _ in range(10)]
    lb = []
    for i in range(10):
        x, t = sp.batch(counter=i)
        lb.append(tb.step(x, t)[0].clone())
    torch.cuda.synchronize()
    assert int(ta.step_dev.item()) == int(tb.step_dev.item()) == 10
    assert torch.equal(torch.cat(la), torch.cat(lb))
    assert torch.equal(ma._plan.flat, mb._plan.flat)
    assert torch.equal(ta.m, tb.m) and torch.equal(ta.v, tb.v)
    assert torch.equal(ma.conv1[2].running_mean, mb.conv1[2].running_mean)
    ta.close()


def _newrale():
    from ecg_denoise_b200.model import ralenet_12leads as TW
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    m.load_state_dict(SW.make_newrale_state_dict(2023), strict=True)
    return m.cuda().train()


def test_finetune_trainer_step_synth_matches_step():
    from ecg_denoise_b200.engine import FineTuneTrainer
    rec, nz = _banks(12, 1, R=3, T=6000)
    sp = _sampler(rec, nz, 16, seed=4)
    models = [_newrale() for _ in range(3)]
    tg = FineTuneTrainer(models[0], use_graph=True)
    te = FineTuneTrainer(models[1], use_graph=False)
    tr = FineTuneTrainer(models[2], use_graph=False)
    steps = 3
    for i in range(steps):
        lg = tg.step_synth(sp)[0].item()
        le = te.step_synth(sp)[0].item()
        x, t = sp.batch(counter=i)
        lr_ = tr.step(x, t)[0].item()
        assert abs(lg - lr_) <= 1e-5 * abs(lr_) and abs(le - lr_) <= 1e-5 * abs(lr_), (i, lg, le, lr_)
    assert int(tg.step_dev.item()) == steps
    # the convolution weight gradients are summed with atomics: Adam can turn their last-bit noise into +-lr moves of
    # elements whose gradient is ~0, so parameters are compared with that bound (steps x lr)
    for t in (tg, te):
        assert float((t.flat - tr.flat).abs().max()) <= steps * 1.05e-3
    # a plain step after step_synth trains on the given batch again, not on the sampler's
    x, t = sp.batch(counter=100)
    out = tg.step(x, t)[3]
    assert torch.equal(tg._x, x)
    assert out.shape == x.shape
    with pytest.raises(ValueError, match="leads"):
        tg.step_synth(_sampler(*_banks(2, 2), 4))
    tg.close()


def test_failures_are_loud():
    from ecg_denoise_b200 import _lib
    rec, nz = _banks(2, 2)
    with pytest.raises(_lib.RalenetError, match="cpu"):
        _sampler(rec.cpu(), nz, 4)
    with pytest.raises(_lib.RalenetError, match="cpu"):
        _sampler(rec, nz.cpu(), 4)
    with pytest.raises(_lib.RalenetError, match="float32"):
        _sampler(rec.double(), nz, 4)
    with pytest.raises(_lib.RalenetError, match="contiguous"):
        _sampler(rec.transpose(1, 2).contiguous().transpose(1, 2), nz, 4)
    with pytest.raises(ValueError):
        _sampler(rec, nz[:, :, :100], 4)
    sp = _sampler(rec, nz, 4)
    good = torch.empty(4, 2, 256, device="cuda")
    with pytest.raises(ValueError, match="shape"):
        sp.fill(torch.empty(4, 2, 128, device="cuda"), good)
    with pytest.raises(_lib.RalenetError):
        sp.fill(good.cpu(), good)
    with pytest.raises(_lib.RalenetError):
        sp.fill(good, good, torch.zeros(1, dtype=torch.int64, device="cuda"))
    # the C entry point rejects what the Python side would have caught
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    a = sp._args
    saved = {f: getattr(a, f) for f, _ in a._fields_}

    def rc(**kw):
        for f, v in saved.items():
            setattr(a, f, v)
        for f, v in kw.items():
            setattr(a, f, v)
        try:
            return lib.ralenet_record_sample(ctypes.byref(a), st)
        finally:
            for f, v in saved.items():
                setattr(a, f, v)

    assert rc(clean_out=good.data_ptr()) == _lib.RL_OK
    assert rc(records=None, clean_out=good.data_ptr()) == _lib.RL_ERR_NULL
    assert rc(clean_out=None) == _lib.RL_ERR_NULL
    for kw in (dict(W=3001), dict(W=2501), dict(leads=13), dict(noise_leads=3), dict(rank=1), dict(world=0),
               dict(n_snr=0), dict(B=100000), dict(stride=0)):
        assert rc(clean_out=good.data_ptr(), **kw) == _lib.RL_ERR_SHAPE, kw
    torch.cuda.synchronize()
