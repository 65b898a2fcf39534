"""GPU checks of the held-out evaluator (evaluate.py; record_enumerate_kernel in csrc/records.cu, eval_window_kernel /
eval_reduce_kernel in csrc/stem_head.cu): the ordered plan against its numpy mirror bit for bit, the windows against
records_to_windows and the SNR mix, the per-level figures against a float64 computation of local_utils/evaluate.py on
the model's own outputs, graph / eager / rank-split agreement, and that evaluating leaves the model and a running
trainer exactly as they were."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import synth_weights as SW
from tests import eval_plan as EP

pytestmark = pytest.mark.gpu
LEVELS = (-4.0, -2.0, 0.0, 2.0, 4.0)


def _banks(leads, noise_leads, R=3, T=3000, N=3, Tn=2500, seed=0):
    rs = np.random.RandomState(seed + 10 * leads + noise_leads)
    rec = rs.standard_normal((R, leads, T)).astype(np.float32) * 2 + 0.7
    nz = rs.standard_normal((N, noise_leads, Tn)).astype(np.float32) * 0.5
    return torch.from_numpy(rec).cuda(), torch.from_numpy(nz).cuda()


def _evaluator(rec, nz, B, **kw):
    from ecg_denoise_b200.evaluate import RecordEvaluator
    return RecordEvaluator(rec, nz, B, **kw)


def _ralenet(seed=2023):
    from ecg_denoise_b200.model import transformer
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(SW.make_state_dict("rw", 1, seed), strict=True)
    return m.cuda()


def _newrale():
    from ecg_denoise_b200.model import ralenet_12leads as TW
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    m.load_state_dict(SW.make_newrale_state_dict(2023), strict=True)
    return m.cuda()


PLAN_CASES = [  # leads, noise leads, R, T, N, Tn, W, stride, B, n_snr, rank, world
    (2, 2, 3, 3000, 3, 2500, 256, 256, 16, 5, 0, 1),       # 33 items: ragged last batch
    (2, 1, 2, 1000, 2, 900, 256, 64, 8, 3, 1, 2),
    (2, 2, 1, 256, 1, 256, 256, 256, 4, 1, 0, 1),          # one window, three empty slots
    (12, 1, 2, 2000, 2, 1500, 256, 200, 6, 2, 2, 3),
    (12, 12, 2, 800, 1, 700, 128, 1, 64, 2, 0, 2),
]


@pytest.mark.parametrize("leads,noise_leads,R,T,N,Tn,W,stride,B,n_snr,rank,world", PLAN_CASES)
def test_plan_matches_the_mirror_and_windows_match_records_to_windows(leads, noise_leads, R, T, N, Tn, W, stride, B,
                                                                      n_snr, rank, world):
    from ecg_denoise_b200 import ops
    from ecg_denoise_b200.inference import records_to_windows
    rec, nz = _banks(leads, noise_leads, R, T, N, Tn)
    seed = 99
    ev = _evaluator(rec, nz, B, window=W, stride=stride, snr_db=LEVELS[:n_snr], seed=seed, rank=rank, world=world)
    assert ev.steps == EP.steps(R, T, W, stride, B, n_snr, world)
    win, _ = records_to_windows(rec, W, stride)
    nper = (T - W) // stride + 1
    levels = torch.tensor(LEVELS[:n_snr], dtype=torch.float32, device="cuda")
    for k in range(ev.steps):
        ev.fill(k)
        meta_ref, lvl_ref = EP.plan(R, T, N, Tn, W, stride, B, n_snr, seed, k, rank, world)
        assert np.array_equal(ev.meta.cpu().numpy().astype(np.int64), meta_ref), k
        assert np.array_equal(ev.level.cpu().numpy().astype(np.int64), lvl_ref), k
        v = torch.from_numpy(lvl_ref >= 0).cuda()
        assert torch.equal(ev.valid, v), k
        tail = torch.nonzero(~v).flatten()
        vi = torch.nonzero(v).flatten()
        mv = meta_ref[lvl_ref >= 0]
        if len(mv):                                        # a rank's last batch may lie wholly past the end
            g = torch.from_numpy(mv[:, 0] * nper + mv[:, 1] // stride).cuda()
            assert torch.equal(ev.clean[vi], win[g]), k
            nref = torch.stack([nz[m[2], :, m[3]:m[3] + W] for m in mv])[:, [l % noise_leads for l in range(leads)]]
            assert torch.equal(ev.noise[vi], nref), k
            snr = levels[torch.from_numpy(lvl_ref[lvl_ref >= 0]).cuda()]
            assert torch.equal(ev.snr[vi], snr), k
            assert torch.equal(ev.noisy[vi], ops.snr_mix(win[g].contiguous(), nref.contiguous(), snr)), k
        else:
            assert len(tail) == B
        assert bool((ev.clean[tail] == 0).all()) and bool((ev.noise[tail] == 0).all()) and bool((ev.snr[tail] == 0).all())


def _reference(ev, model, n_snr):
    """per-level (count, mean snr_in, mean snr_out, mean rmse) in float64 from model(x) under torch.no_grad() in eval
    mode, on the evaluator's own noisy windows, batch by batch."""
    was = model.training
    model.eval()
    sums = np.zeros((n_snr, 4))
    with torch.no_grad():
        for k in range(ev.steps):
            ev.fill(k)
            out = model(ev.noisy)
            v = ev.valid
            assert bool(torch.isfinite(out[v]).all())          # the zero windows of the tail stay in their slots
            y, x, p = (t[v].double().flatten(1) for t in (ev.clean, ev.noisy, out))
            sy = (y ** 2).sum(1)
            snr_in = 10 * torch.log10(sy / ((y - x) ** 2).sum(1))
            snr_out = 10 * torch.log10(sy / ((y - p) ** 2).sum(1))
            rmse = torch.sqrt(((y - p) ** 2).mean(1))
            lvl = ev.level[v].long()
            for l in range(n_snr):
                s = lvl == l
                sums[l] += [float(s.sum()), float(snr_in[s].sum()), float(snr_out[s].sum()), float(rmse[s].sum())]
    model.train(was)
    return sums


def _assert_matches(res, ev, sums, rel=1e-6):
    for l, lv in enumerate(ev.levels):
        n = sums[l, 0]
        assert res.count[lv] == n
        for got, s in ((res.snr_in[lv], sums[l, 1]), (res.snr_out[lv], sums[l, 2]), (res.rmse[lv], sums[l, 3])):
            ref = s / n
            assert abs(got - ref) <= rel * abs(ref) + 1e-9, (lv, got, ref)
        assert res.snr_imp[lv] == res.snr_out[lv] - res.snr_in[lv]


def test_per_level_means_match_float64_on_the_model_outputs():
    rec, nz = _banks(2, 1, R=3, T=5000)
    ev = _evaluator(rec, nz, 48, stride=200, seed=5)          # 3 * 23 * 5 = 345 items: a ragged last batch
    assert ev.n_items % ev.B != 0
    model = _ralenet()
    res = ev.run(model)
    sums = _reference(ev, model, len(LEVELS))
    assert sum(res.count.values()) == ev.n_items
    _assert_matches(res, ev, sums)
    assert res.acc.dtype == torch.float64 and tuple(res.acc.shape) == (len(LEVELS), 4)


def test_graph_and_eager_runs_are_bit_identical_and_repeatable():
    rec, nz = _banks(2, 2, R=2, T=6000)
    ev = _evaluator(rec, nz, 40, stride=128, seed=3)
    model = _ralenet()
    a = ev.run(model, use_graph=True).acc.clone()
    b = ev.run(model, use_graph=True).acc.clone()
    c = ev.run(model, use_graph=False).acc.clone()
    assert torch.equal(a, b) and torch.equal(a, c)
    assert int(ev.counter.item()) == ev.steps


def test_rank_slices_sum_to_the_single_process_result():
    rec, nz = _banks(2, 1, R=3, T=4000)
    model = _ralenet()
    whole = _evaluator(rec, nz, 32, stride=100, seed=9).run(model).acc.clone()
    world = 3
    parts = [_evaluator(rec, nz, 16, stride=100, seed=9, rank=r, world=world).run(model).acc.clone()
             for r in range(world)]
    total = sum(parts[1:], parts[0].clone())
    assert torch.equal(total[:, 0], whole[:, 0])
    assert float(((total - whole).abs() / whole.abs().clamp_min(1e-300)).max()) <= 1e-12


def test_run_leaves_the_model_untouched():
    rec, nz = _banks(2, 2)
    ev = _evaluator(rec, nz, 24, stride=256)
    model = _ralenet().train()
    model.inference_precision = "fp32"
    model.dtransformer2.eval()                                # a mixed mode is restored module by module
    bn = model.conv1[2]
    with torch.no_grad():
        bn.running_mean.uniform_(-0.1, 0.1)
        bn.running_var.uniform_(0.5, 1.5)
    model(rec[:1, :, :256].contiguous())                      # build the flat parameter plan
    before = [model._plan.flat.clone(), bn.running_mean.clone(), bn.running_var.clone(),
              bn.num_batches_tracked.clone()]
    modes = [m.training for m in model.modules()]
    for use_graph in (True, False):
        ev.run(model, precision="tf32", use_graph=use_graph)
        after = [model._plan.flat, bn.running_mean, bn.running_var, bn.num_batches_tracked]
        assert all(torch.equal(u, w) for u, w in zip(before, after))
        assert [m.training for m in model.modules()] == modes
        assert model.inference_precision == "fp32"
        assert all(p.grad is None for p in model.parameters())


def test_run_between_trainer_replays_does_not_change_the_trajectory():
    from ecg_denoise_b200.engine import FusedTrainer
    from ecg_denoise_b200.record_sampler import RecordSampler
    rec, nz = _banks(2, 1, R=4, T=20000)
    hold, hnz = _banks(2, 1, R=2, T=6000, seed=5)
    sp = RecordSampler(rec, nz, 64, seed=8)
    ev = _evaluator(hold, hnz, 64, stride=128)
    ma, mb = _ralenet().train(), _ralenet().train()
    ta = FusedTrainer(ma, use_graph=True, deterministic=True)
    tb = FusedTrainer(mb, use_graph=True, deterministic=True)
    la, lb, graphs = [], [], []
    for i in range(8):
        la.append(ta.step_synth(sp)[0].clone())
        lb.append(tb.step_synth(sp)[0].clone())
        graphs.append(ta.graph)
        if i in (2, 5):
            res = ev.run(ma, use_graph=(i == 2))
            assert sum(res.count.values()) == ev.n_items
            assert ma.training
    torch.cuda.synchronize()
    assert all(g is graphs[0] for g in graphs)                # the trainer's captured step was kept
    assert torch.equal(torch.cat(la), torch.cat(lb))
    assert torch.equal(ma._plan.flat, mb._plan.flat)
    assert torch.equal(ma.conv1[2].running_mean, mb.conv1[2].running_mean)
    assert torch.equal(ma.conv1[2].num_batches_tracked, mb.conv1[2].num_batches_tracked)
    ta.close()
    tb.close()


def test_tf32_is_within_a_hundredth_of_a_db_of_fp32():
    rec, nz = _banks(2, 1, R=3, T=8000)
    ev = _evaluator(rec, nz, 128, stride=128, seed=4)
    model = _ralenet()
    f = ev.run(model, precision="fp32")
    t = ev.run(model, precision="tf32")
    assert model.inference_precision == "fp32"
    for lv in ev.levels:
        assert f.count[lv] == t.count[lv]
        assert abs(f.snr_out[lv] - t.snr_out[lv]) <= 0.01, lv
        assert f.snr_in[lv] == t.snr_in[lv]


def test_newrale_on_a_twelve_lead_bank():
    rec, nz = _banks(12, 1, R=2, T=3000)
    ev = _evaluator(rec, nz, 16, stride=256, snr_db=(-2, 0, 3))
    model = _newrale().train()
    res = ev.run(model)
    assert model.training
    sums = _reference(ev, model, 3)
    assert sum(res.count.values()) == ev.n_items
    _assert_matches(res, ev, sums)


def test_failures_are_loud():
    from ecg_denoise_b200 import _lib
    rec2, nz2 = _banks(2, 2)
    rec12, nz12 = _banks(12, 1, R=2)
    with pytest.raises(ValueError, match="leads"):
        _evaluator(rec12, nz12, 4).run(_ralenet())
    with pytest.raises(ValueError, match="leads"):
        _evaluator(rec2, nz2, 4).run(_newrale())
    with pytest.raises(TypeError):
        _evaluator(rec2, nz2, 4).run(torch.nn.Conv1d(2, 2, 3).cuda())
    with pytest.raises(ValueError):
        _evaluator(rec2, nz2, 4).run(_ralenet(), precision="fp16")
    with pytest.raises(_lib.RalenetError, match="float32"):
        _evaluator(rec2.double(), nz2, 4)
    # the C entry points reject bad arguments before any launch
    ev = _evaluator(rec2, nz2, 4)
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rc(fn, a, **kw):
        saved = {f: getattr(a, f) for f, _ in a._fields_}
        try:
            for f, v in kw.items():
                setattr(a, f, v)
            return getattr(lib, fn)(ctypes.byref(a), st)
        finally:
            for f, v in saved.items():
                setattr(a, f, v)

    assert rc("ralenet_record_enumerate", ev._args) == _lib.RL_OK
    for kw in (dict(records=None), dict(level=None), dict(clean_out=None), dict(snr_levels=None)):
        assert rc("ralenet_record_enumerate", ev._args, **kw) == _lib.RL_ERR_NULL, kw
    for kw in (dict(W=3001), dict(W=2501), dict(leads=13), dict(noise_leads=3), dict(rank=1), dict(rank=-1),
               dict(world=0), dict(n_snr=0), dict(B=0), dict(stride=0), dict(T=2 ** 31), dict(Tn=2 ** 31),
               dict(R=2 ** 31 - 1, n_snr=2 ** 31 - 1)):
        assert rc("ralenet_record_enumerate", ev._args, **kw) == _lib.RL_ERR_SHAPE, kw
    m = ev._margs
    m.pred = ev.noisy.data_ptr()
    for kw in (dict(clean=None), dict(pred=None), dict(level=None), dict(partials=None), dict(acc=None)):
        assert rc("ralenet_eval_metrics", m, **kw) == _lib.RL_ERR_NULL, kw
    for kw in (dict(B=0), dict(per=0), dict(n_snr=0)):
        assert rc("ralenet_eval_metrics", m, **kw) == _lib.RL_ERR_SHAPE, kw
    torch.cuda.synchronize()
