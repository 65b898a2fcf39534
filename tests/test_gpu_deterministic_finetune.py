"""Deterministic mode of the 12-lead fine-tune on the GPU: the deterministic convolution backward
(ralenet_conv1d_bwd_det) against the fp64 oracle and the atomic path, bit identity of FineTuneTrainer(deterministic=
True) and of the drop-in newrale under torch.use_deterministic_algorithms(True) across schedules, a bit-identical
trajectory, and accuracy on poisoned workspaces and slabs.

Bit identity holds for a fixed build, model, batch shape and kernel-selection switches (ralenet_set_conv_mma
included), so every comparison below is between runs with the same switches."""
import ctypes
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import ralenet_oracle as O
from oracle import synth_weights as SW
from tests.common import check_packed, rel_rms_err, switches, unpack_golden

pytestmark = pytest.mark.gpu
RTOL = 1e-3
POISON = {"nan": 0xFF, "finite": 0x7E}
LAYERS = [(12, 6, True), (6, 2, True), (2, 6, True), (6, 12, False)]     # (Cin, Cout, LeakyReLU) of newrale
# kernel family -> (L, ralenet_set_conv_mma): tensor-core kernels, scalar kernels by switch, scalar kernels because L
# is not a multiple of 32
FAMILIES = {"mma": (256, 1), "fma": (256, 0), "fma_ragged": (200, 1)}


@contextmanager
def torch_deterministic(warn_only=False):
    state = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(state[0], warn_only=state[1])


@contextmanager
def conv_mma(on):
    from ecg_denoise_b200 import _lib
    prev = _lib.load().ralenet_set_conv_mma(on)
    try:
        yield
    finally:
        _lib.load().ralenet_set_conv_mma(prev)


def _equal(a, b, what):
    for i, (u, v) in enumerate(zip(a, b)):
        assert torch.equal(u, v), f"{what}: item {i} differs (max |d| = {(u - v).abs().max().item():.3e})"


def _profiled(fn):
    from ecg_denoise_b200 import _lib
    lib = _lib.load()
    _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    try:
        return fn()
    finally:
        n_max = 8192
        labels = ctypes.create_string_buffer(n_max * 48)
        ms = (ctypes.c_float * n_max)()
        lib.ralenet_profile_end(labels, 48, ms, n_max)


def _side_load():
    """concurrent elementwise work on another stream: takes SMs away at unpredictable moments."""
    side = torch.cuda.Stream()
    z = torch.rand(1 << 24, device="cuda")
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(40):
            z.mul_(1.0000001).add_(1e-7)
    return side


def _newrale():
    from ecg_denoise_b200.model import ralenet_12leads as TW
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    m.load_state_dict(SW.make_newrale_state_dict(2023), strict=True)
    return m.cuda().train()


def _inputs12(B, L=256, seed=5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, 12, L, device="cuda", generator=g), torch.randn(B, 12, L, device="cuda", generator=g)


# ------------------------------------------------------------------------------------------------------------------
# 1. the C entry point, layer by layer

def _conv_bwd(ops, B, L, ci, co, act, x, w, b, dy, dx, d_w, d_b, slab=None):
    from ecg_denoise_b200 import _lib
    a = ops._fill("rl_conv_bwd_args", B=B, L=L, Cin=ci, Cout=co, K=13, act=int(act), slope=0.01, dy=dy, x=x, w=w, b=b,
                  dx=ops._p(dx), d_w=ops._p(d_w), d_b=ops._p(d_b))
    if slab is None:
        _lib.call("ralenet_conv1d_bwd", a, ops._stream())
    else:
        ops.conv1d_bwd_det(a, slab)
    return a


@pytest.mark.parametrize("B", [1, 37, 1280])
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("ci,co,act", LAYERS + [(12, 6, False), (6, 12, True)])
def test_conv_bwd_det_vs_oracle_and_atomic_path(ci, co, act, family, B):
    from ecg_denoise_b200 import _lib, ops
    L, mma = FAMILIES[family]
    rs = np.random.RandomState(1000 + 10 * ci + co)
    f = lambda *s: torch.from_numpy(rs.standard_normal(s)).cuda()
    w64, b64 = f(co, ci, 13) * (13 * ci) ** -0.5, 0.1 * f(co)
    x64, dy64 = f(B, ci, L), f(B, co, L)
    c = O.conv1d_fwd(x64, w64, b64)
    dc = dy64 * torch.where(c > 0, torch.ones_like(c), torch.full_like(c, 0.01)) if act else dy64
    _, dw_ref, db_ref = O.conv1d_bwd(dc, x64, w64)
    x, w, b, dy = (t.float().contiguous() for t in (x64, w64, b64, dy64))
    g0w, g0b = f(co, ci, 13).float(), f(co).float()       # a gradient that already holds something
    nbytes = int(_lib.load().ralenet_conv1d_slab_bytes(B, ci, co, 13))
    slab = torch.empty(nbytes // 4, device="cuda")
    with conv_mma(mma):
        dx_at, dw_at, db_at = torch.empty_like(x), torch.zeros_like(w), torch.zeros_like(b)
        _conv_bwd(ops, B, L, ci, co, act, x, w, b, dy, dx_at, dw_at, db_at)

        def det(byte, gw, gb, dx=True, db=True):
            if byte is None:
                slab.zero_()
            else:
                slab.view(torch.uint8).fill_(byte)
            out = (torch.empty_like(x) if dx else None, gw.clone(), gb.clone() if db else None)
            _conv_bwd(ops, B, L, ci, co, act, x, w, b, dy, *out, slab=slab)
            return out

        dx_d, dw_d, db_d = det(None, torch.zeros_like(w), torch.zeros_like(b))
        for byte in POISON.values():
            _equal((dx_d, dw_d, db_d), det(byte, torch.zeros_like(w), torch.zeros_like(b)), f"poison {byte:#x}")
        # += onto a non-zero gradient: the window sum is added with one fp32 add per element
        _, dw_acc, db_acc = det(POISON["nan"], g0w, g0b)
        _equal((dw_acc, db_acc), (g0w + dw_d, g0b + db_d), "accumulate")
        # NULL dx and NULL d_b
        dxn, dw_n, dbn = det(POISON["nan"], torch.zeros_like(w), None, dx=False, db=False)
        assert dxn is None and dbn is None
        _equal((dw_n,), (dw_d,), "NULL dx / d_b")
        # a short or missing slab is refused before anything is launched
        a = ops._fill("rl_conv_bwd_args", B=B, L=L, Cin=ci, Cout=co, K=13, act=int(act), slope=0.01, dy=dy, x=x, w=w,
                      b=b, dx=None, d_w=dw_n, d_b=None)
        with pytest.raises(_lib.RalenetError):
            ops.conv1d_bwd_det(a, slab[:-1])
        with pytest.raises(_lib.RalenetError):
            _lib.check(_lib.load().ralenet_conv1d_bwd_det(ctypes.byref(a), None, nbytes, ops._stream()))
    torch.cuda.synchronize()
    assert torch.equal(dx_d, dx_at), "dx is a plain store in both modes"
    tag = f"{ci}to{co}/act{int(act)}/{family}/B{B}"
    for name, got, ref in (("dw", dw_d, dw_ref), ("db", db_d, db_ref)):
        e = rel_rms_err(got.double().cpu().numpy(), ref.cpu().numpy())
        assert e <= RTOL, f"{tag}/{name}: {e:.3e} vs the fp64 oracle"
    for name, got, ref in (("dw", dw_d, dw_at), ("db", db_d, db_at)):
        e = rel_rms_err(got.double().cpu().numpy(), ref.double().cpu().numpy())
        assert e <= 2e-5, f"{tag}/{name}: {e:.3e} vs the atomic path"


# ------------------------------------------------------------------------------------------------------------------
# 2. bit identity across schedules

def _trainer_state(tr, m):
    bn = m.rale.conv1[2]
    plan = m.rale._plan
    return (tr._res[0].clone(), tr._da1.clone(), tr.flat_grad.clone(), plan.bn_stats[32:48].clone(), tr.flat.clone(),
            tr.m.clone(), tr.v.clone(), tr.step_dev.clone(), bn.running_mean.clone(), bn.running_var.clone(),
            bn.num_batches_tracked.clone())


def _trainer_run(x, t, graph=False, wrap=None, before=None):
    from ecg_denoise_b200.engine import FineTuneTrainer
    m = _newrale()
    tr = FineTuneTrainer(m, lr=1e-3, use_graph=graph, deterministic=True)
    tr._prepare(x.shape, x.device)
    side = before() if before is not None else None
    (wrap or (lambda fn: fn()))(lambda: tr.step(x, t))
    if side is not None:
        torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    out = _trainer_state(tr, m)
    tr.close()
    return out


def _dropin_run(x, t, wrap=None, before_backward=None):
    """drop-in step under the torch flag: model(x), F.mse_loss, backward(), torch.optim.Adam."""
    m = _newrale()
    convs = [m.conv1, m.conv2, m.conv3, m.conv4]
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-3)

    def step():
        with torch_deterministic():
            xg = x.clone().requires_grad_(True)
            loss = torch.nn.functional.mse_loss(m(xg), t)
            side = before_backward() if before_backward is not None else None
            loss.backward()
            if side is not None:
                torch.cuda.current_stream().wait_stream(side)
            grads = [p.grad.clone() for c in convs for p in (c.weight, c.bias)]
            opt.step()
        return loss.detach().clone(), xg.grad.clone(), grads
    loss, dx, grads = (wrap or (lambda fn: fn()))(step)
    torch.cuda.synchronize()
    bn = m.rale.conv1[2]
    return (loss, dx, *grads, m.rale._plan.bn_stats[32:48].clone(),
            *[p.detach().clone() for c in convs for p in (c.weight, c.bias)],
            bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone())


@pytest.mark.parametrize("mma", [1, 0])
@pytest.mark.parametrize("mode", ["default", "reg2", "mma"])
def test_finetune_trainer_is_bit_identical_across_schedules(mode, mma):
    x, t = _inputs12(37, seed=21)
    with switches(mode), conv_mma(mma):
        ref = _trainer_run(x, t)
        _equal(ref, _trainer_run(x, t), f"{mode}/{mma}: fresh trainer")
        g1 = _trainer_run(x, t, graph=True)
        _equal(ref, g1, f"{mode}/{mma}: graph vs eager")
        _equal(g1, _trainer_run(x, t, graph=True), f"{mode}/{mma}: graph vs graph")
        _equal(ref, _trainer_run(x, t, wrap=_profiled), f"{mode}/{mma}: serial path")
        _equal(ref, _trainer_run(x, t, before=_side_load), f"{mode}/{mma}: concurrent work")
    assert int(ref[7].item()) == 1


@pytest.mark.parametrize("mma", [1, 0])
@pytest.mark.parametrize("mode", ["default", "reg2", "mma"])
def test_dropin_newrale_is_bit_identical_under_the_torch_flag(mode, mma):
    x, t = _inputs12(37, seed=22)
    with switches(mode), conv_mma(mma):
        ref = _dropin_run(x, t)
        _equal(ref, _dropin_run(x, t), f"{mode}/{mma}: fresh model")
        _equal(ref, _dropin_run(x, t, wrap=_profiled), f"{mode}/{mma}: serial path")
        _equal(ref, _dropin_run(x, t, before_backward=_side_load), f"{mode}/{mma}: concurrent work")


# ------------------------------------------------------------------------------------------------------------------
# 3. trajectory on a 12-lead record bank

def _sampler12(B=16):
    from ecg_denoise_b200.record_sampler import RecordSampler
    rs = np.random.RandomState(12)
    rec = torch.from_numpy(rs.standard_normal((3, 12, 6000)).astype(np.float32) * 2 + 0.7).cuda()
    nz = torch.from_numpy(rs.standard_normal((3, 1, 2500)).astype(np.float32) * 0.5).cuda()
    return RecordSampler(rec, nz, B, seed=4)


def test_graphed_trajectory_is_bit_identical_and_step_synth_equals_step():
    from ecg_denoise_b200.engine import FineTuneTrainer
    sp = _sampler12()
    runs = []
    for _ in range(2):
        m = _newrale()
        tr = FineTuneTrainer(m, use_graph=True, deterministic=True)
        losses = [tr.step_synth(sp)[0].clone() for _ in range(20)]
        torch.cuda.synchronize()
        runs.append((torch.cat(losses), *_trainer_state(tr, m)[2:]))
        tr.close()
    assert int(runs[0][6].item()) == 20
    _equal(runs[0], runs[1], "20 graphed step_synth steps")
    # step_synth (the draw inside the graph) and step on the same batches: bit-equal, where the default mode needs a
    # steps x lr bound on the parameters
    te, tr_ = FineTuneTrainer(_newrale(), deterministic=True), FineTuneTrainer(_newrale(), deterministic=True)
    tg = FineTuneTrainer(_newrale(), use_graph=True, deterministic=True)
    for i in range(3):
        lg, le = tg.step_synth(sp)[0].clone(), te.step_synth(sp)[0].clone()
        x, t = sp.batch(counter=i)
        lr_ = tr_.step(x, t)[0].clone()
        _equal((lg, le), (lr_, lr_), f"loss of step {i}")
    torch.cuda.synchronize()
    _equal((tg.flat, te.flat, tg.m, te.v), (tr_.flat, tr_.flat, tr_.m, tr_.v), "parameters after 3 steps")
    tg.close()


# ------------------------------------------------------------------------------------------------------------------
# 4. accuracy on poisoned workspaces and slabs

def _poison_finetune(tr, x, byte):
    tr._prepare(x.shape, x.device)
    tr._ws.fill_(byte)
    tr._loss_partials.view(torch.uint8).fill_(byte)
    for s in tr._slabs.values():
        s.view(torch.uint8).fill_(byte)
    return len(tr._slabs)


@pytest.mark.parametrize("pattern", list(POISON))
@pytest.mark.parametrize("graph", [False, True])
def test_det_finetune_trainer_meets_the_golden_adam_trajectory(golden, graph, pattern):
    from ecg_denoise_b200.engine import FineTuneTrainer
    sd = SW.make_newrale_state_dict(2023)
    x = torch.from_numpy(golden["x12"]).cuda()
    tgt = torch.from_numpy(golden["target12"]).cuda()
    m = _newrale()
    tr = FineTuneTrainer(m, lr=0.001, use_graph=graph, deterministic=True)
    assert _poison_finetune(tr, x, POISON[pattern]) == 4
    losses = [tr.step(x, tgt)[0].item() for _ in range(3)]
    ref = golden["newrale/adam_losses64"]
    assert np.allclose(losses, ref, rtol=2e-4), (losses, ref)
    names = [str(n) for n in golden["newrale/grad_names"]]
    params = dict(m.named_parameters())
    gold = unpack_golden(names, golden["newrale/adam_params"], {n: tuple(sd[n].shape) for n in names})
    for n in names:
        check_packed(params[n].detach(), gold[n], RTOL, f"det_finetune/graph{int(graph)}/{pattern}/param/{n}")
    assert int(m.rale.conv1[2].num_batches_tracked.item()) == 3 + 3
    for n, p in params.items():
        if n.startswith("rale."):
            assert torch.equal(p.detach().cpu(), sd[n]), n
    tr.close()


@pytest.fixture
def poison_dropin(monkeypatch):
    """poison(byte): every workspace the drop-in forward leases and every convolution slab is filled with `byte`
    first.  Returns the list of poisoned buffer sizes."""
    from ecg_denoise_b200 import engine, ops
    lease_ws, conv1d_slab = engine._lease_ws, ops.conv1d_slab
    state = {"byte": None}
    hits = []

    def leased(plan, nbytes, device):
        lease = lease_ws(plan, nbytes, device)
        lease.buf.fill_(state["byte"])
        hits.append(("ws", nbytes))
        return lease

    def slab(*args):
        s = conv1d_slab(*args)
        s.view(torch.uint8).fill_(state["byte"])
        hits.append(("slab", s.numel()))
        return s

    monkeypatch.setattr(engine, "_lease_ws", leased)
    monkeypatch.setattr(ops, "conv1d_slab", slab)

    def set_pattern(byte):
        state["byte"] = byte
        return hits
    return set_pattern


@pytest.mark.parametrize("pattern", list(POISON))
def test_det_dropin_newrale_meets_the_golden_gradients(golden, poison_dropin, pattern):
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.engine import workspace_bytes
    hits = poison_dropin(POISON[pattern])
    sd = SW.make_newrale_state_dict(2023)
    m = _newrale()
    x = torch.from_numpy(golden["x12"]).cuda().requires_grad_(True)
    tgt = torch.from_numpy(golden["target12"]).cuda()
    with torch_deterministic():
        y = m(x)
        torch.nn.functional.mse_loss(y, tgt).backward()
    torch.cuda.synchronize()
    B, _, L = x.shape
    assert m.rale._plan.last_ws_bytes == workspace_bytes(B, L, True, _lib.RL_NET_DETERMINISTIC)
    assert sum(1 for k, _ in hits if k == "slab") == 4 and any(k == "ws" for k, _ in hits)
    assert rel_rms_err(y.detach().double().cpu().numpy(), golden["newrale/train_out64"]) <= RTOL
    assert rel_rms_err(x.grad.double().cpu().numpy(), golden["newrale/dx64"]) <= RTOL
    names = [str(n) for n in golden["newrale/grad_names"]]
    params = dict(m.named_parameters())
    gold = unpack_golden(names, golden["newrale/grads"], {n: tuple(sd[n].shape) for n in names})
    for n in names:
        check_packed(params[n].grad, gold[n], RTOL, f"det_newrale/{pattern}/grad/{n}")
    for n, p in params.items():
        if n.startswith("rale."):
            assert p.grad is None, n


def test_det_dropin_newrale_at_config3_shape_vs_oracle(poison_dropin):
    """1280 windows of 12 x 256 under the torch flag on NaN-poisoned buffers, against the fp64 oracle, with the bounds
    of test_gpu_net.py::test_newrale_at_config3_shape_vs_oracle (dx: a few LeakyReLU slopes decided differently in
    fp32 and fp64 move single samples by O(1), so dx is bounded element-wise for all but 2e-3 of the elements, in L2
    and per median window)."""
    from ecg_denoise_b200 import synth
    hits = poison_dropin(POISON["nan"])
    sd = SW.make_newrale_state_dict(2023)
    m = _newrale()
    B = 1280
    noisy, clean = synth.make_batch(128, 12, 256, seed=12, kind="bw", snr_db=2.0)
    gains = np.random.RandomState(2).uniform(0.6, 1.4, size=(10, 1, 1, 1)).astype(np.float32)
    x = torch.from_numpy((noisy[None] * gains).reshape(B, 12, 256))
    tgt = torch.from_numpy((clean[None] * gains).reshape(B, 12, 256))
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    out_ref, ctx = O.newrale_fwd(x.double(), sd64, training=True)[:2]
    loss_ref, dout = O.mse_loss_fwd_bwd(out_ref, tgt.double())
    dx_ref, grads = O.newrale_bwd(dout, ctx, sd64)
    xc = x.cuda().requires_grad_(True)
    with torch_deterministic():
        y = m(xc)
        loss = torch.nn.functional.mse_loss(y, tgt.cuda())
        loss.backward()
    torch.cuda.synchronize()
    assert sum(1 for k, _ in hits if k == "slab") == 4
    assert rel_rms_err(y.detach().double().cpu().numpy(), out_ref.numpy()) <= RTOL
    got, ref = xc.grad.detach().double().cpu().numpy(), dx_ref.numpy()
    rms = np.sqrt((ref * ref).mean())
    bad = np.abs(got - ref) > RTOL * (np.abs(ref) + rms)
    assert bad.mean() < 2e-3, bad.mean()
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 2e-2
    assert np.median((np.abs(got - ref) / (np.abs(ref) + rms)).reshape(B, -1).max(1)) < RTOL
    assert abs(loss.item() - loss_ref.item()) <= 1e-4 * abs(loss_ref.item())
    for n, p in m.named_parameters():
        if p.requires_grad:
            e = rel_rms_err(p.grad.double().cpu().numpy(), grads[n].numpy())
            assert e <= RTOL, f"{n}: {e:.3e}"
        else:
            assert p.grad is None, n


# ------------------------------------------------------------------------------------------------------------------
# 5. the torch flag

def test_torch_flag_selects_the_deterministic_finetune_and_guards_a_mixed_conv():
    from ecg_denoise_b200 import ops
    from ecg_denoise_b200.engine import FineTuneTrainer
    x, t = _inputs12(8, seed=23)
    with torch_deterministic():
        tr = FineTuneTrainer(_newrale())
        assert tr.deterministic
        loss = tr.step(x, t)[0]            # no guard: the trainer is deterministic
    assert torch.isfinite(loss).all()
    assert not FineTuneTrainer(_newrale()).deterministic
    w = torch.randn(6, 12, 13, device="cuda", requires_grad=True)
    b = torch.randn(6, device="cuda", requires_grad=True)
    y = ops.Conv1dFn.apply(x, w, b, True, 0.01)          # forward without the flag: atomic backward
    with torch_deterministic():
        with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
            y.backward(torch.ones_like(y), retain_graph=True)
    with torch_deterministic(warn_only=True):
        with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
            y.backward(torch.ones_like(y))
    assert w.grad is not None and torch.isfinite(w.grad).all()
    assert not torch.are_deterministic_algorithms_enabled()
