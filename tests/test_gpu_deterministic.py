"""Deterministic mode (RL_NET_DETERMINISTIC) on the GPU: bit-identical results across schedules, accuracy against the
reference golden vectors, a bit-identical Adam trajectory, and torch.use_deterministic_algorithms(True).

Bit identity holds for a fixed build, model, batch shape and kernel-selection switches, so every comparison below is
between runs with the same switches."""
import ctypes
import os
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import synth_weights as SW
from tests.common import CASES, check_packed, rel_rms_err, unpack_golden

pytestmark = pytest.mark.gpu
RTOL = 1e-3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def golden_det():
    return np.load(os.path.join(ROOT, "tests", "golden", "ralenet_golden.npz"), allow_pickle=False)


@contextmanager
def torch_deterministic(warn_only=False):
    state = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(state[0], warn_only=state[1])


@contextmanager
def switches(mode):
    """kernel-selection switches: 'default', 'reg2' (register-tile GEMMs for every group), 'mma' (mma.sync GEMMs)."""
    from ecg_denoise_b200 import _lib
    lib = _lib.load()
    prev_reg, prev_umma = lib.ralenet_set_wgrad_reg(1), lib.ralenet_set_wgrad_umma(1)
    if mode == "reg2":
        lib.ralenet_set_wgrad_reg(2)
    elif mode == "mma":
        lib.ralenet_set_wgrad_reg(0)
        lib.ralenet_set_wgrad_umma(0)
    try:
        yield
    finally:
        lib.ralenet_set_wgrad_reg(prev_reg)
        lib.ralenet_set_wgrad_umma(prev_umma)


MODELS = {"rw_le_256": ("rw", 1, 256, 256), "rw_le_515": ("rw", 1, 515, 256), "nra512": ("nra", 1, 48, 512)}


def _model(variant, le):
    from ecg_denoise_b200.model import raletransformer, transformer
    m = raletransformer.ralenet() if variant == "nra" else transformer.ralenet(high_level_enhence=bool(le))
    m.load_state_dict(SW.make_state_dict(variant, le, 2023), strict=True)
    return m.cuda().train()


def _inputs(B, L0, seed=5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, 2, L0, device="cuda", generator=g)
    t = torch.randn(B, 2, L0, device="cuda", generator=g)
    return x, t


def _dropin_backward(m, x, t, before_backward=None):
    """deterministic drop-in forward + backward (torch flag on): returns (loss, dx, flat_grad, BN backward sums)."""
    from ecg_denoise_b200 import ops
    with torch_deterministic():
        xg = x.clone().requires_grad_(True)
        m._plan.flat_grad.zero_() if m._plan.flat_grad is not None else None
        y = m(xg)
        loss, dout, _, _ = ops.mse_loss_metrics(y.detach(), t)
        if before_backward is not None:
            before_backward()
        y.backward(dout)
    torch.cuda.synchronize()
    return loss.clone(), xg.grad.clone(), m._plan.flat_grad.clone(), m._plan.bn_stats[32:48].clone()


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


@pytest.mark.parametrize("mode", ["default", "reg2", "mma"])
@pytest.mark.parametrize("tag", list(MODELS))
def test_dropin_backward_is_bit_identical_across_schedules(tag, mode):
    variant, le, B, L0 = MODELS[tag]
    x, t = _inputs(B, L0)
    with switches(mode):
        ref = _dropin_backward(_model(variant, le), x, t)
        _equal(ref, _dropin_backward(_model(variant, le), x, t), f"{tag}/{mode}: fresh model")
        # the profiler's serial path: every kernel, weight-gradient GEMMs and reductions included, on one stream
        _equal(ref, _profiled(lambda: _dropin_backward(_model(variant, le), x, t)), f"{tag}/{mode}: serial path")
        # concurrent elementwise work on another stream takes SMs away at unpredictable moments
        side = torch.cuda.Stream()
        z = torch.rand(1 << 24, device="cuda")

        def load():
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(40):
                    z.mul_(1.0000001).add_(1e-7)
        got = _dropin_backward(_model(variant, le), x, t, before_backward=load)
        torch.cuda.current_stream().wait_stream(side)
        _equal(ref, got, f"{tag}/{mode}: concurrent work")


@pytest.mark.parametrize("mode", ["default", "reg2", "mma"])
@pytest.mark.parametrize("tag", list(MODELS))
def test_fused_trainer_graph_replay_equals_eager_step(tag, mode):
    from ecg_denoise_b200.engine import FusedTrainer
    variant, le, B, L0 = MODELS[tag]
    x, t = _inputs(B, L0, seed=9)
    res = []
    with switches(mode):
        for graph in (False, True, True):
            m = _model(variant, le)
            tr = FusedTrainer(m, lr=1e-3, use_graph=graph, deterministic=True)
            loss = tr.step(x, t)[0]
            torch.cuda.synchronize()
            res.append((loss.clone(), m._plan.flat_grad.clone(), m._plan.flat.clone(), tr.m.clone(), tr.v.clone()))
            tr.close()
    _equal(res[0], res[1], f"{tag}/{mode}: graph vs eager")
    _equal(res[1], res[2], f"{tag}/{mode}: graph vs graph")


@pytest.mark.parametrize("tag", list(CASES))
def test_deterministic_gradients_meet_reference_golden(golden_det, tag):
    variant, le, seed, xk, tk = CASES[tag]
    from ecg_denoise_b200.model import raletransformer, transformer
    m = raletransformer.ralenet() if variant == "nra" else transformer.ralenet(high_level_enhence=bool(le))
    sd = SW.make_state_dict(variant, le, seed)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    x = torch.from_numpy(golden_det[xk]).cuda().requires_grad_(True)
    tgt = torch.from_numpy(golden_det[tk]).cuda()
    with torch_deterministic():
        y = m(x)
        loss = torch.nn.functional.mse_loss(y, tgt)
        loss.backward()
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.engine import workspace_bytes
    assert m._plan.last_ws_bytes == workspace_bytes(x.shape[0], x.shape[2], True, _lib.RL_NET_DETERMINISTIC)
    assert rel_rms_err(y.detach().double().cpu().numpy(), golden_det[f"{tag}/train_out64"]) <= RTOL
    assert rel_rms_err(x.grad.double().cpu().numpy(), golden_det[f"{tag}/dx64"]) <= RTOL
    names = [str(n) for n in golden_det[f"{tag}/grad_names"]]
    params = dict(m.named_parameters())
    gold = unpack_golden(names, golden_det[f"{tag}/grads"], {n: tuple(sd[n].shape) for n in names})
    for n in names:
        check_packed(params[n].grad, gold[n], RTOL, f"{tag}/det_grad/{n}")


def test_adam_trajectory_is_bit_identical():
    from ecg_denoise_b200.engine import FusedTrainer
    from ecg_denoise_b200.synth_device import DeviceSynth
    runs = []
    for _ in range(2):
        m = _model("rw", 1)
        tr = FusedTrainer(m, lr=1e-3, use_graph=True, deterministic=True)
        sy = DeviceSynth(256, 2, 256, seed=11, kind="emb", snr_db=-4.0)
        losses = [tr.step_synth(sy)[0].clone() for _ in range(20)]
        torch.cuda.synchronize()
        runs.append((torch.cat(losses), m._plan.flat.clone(), tr.m.clone(), tr.v.clone(), tr.step_dev.clone(),
                     m.conv1[2].running_mean.clone(), m.conv1[2].running_var.clone()))
        tr.close()
    assert int(runs[0][4].item()) == 20
    _equal(runs[0], runs[1], "20 graphed step_synth steps")


def test_torch_flag_selects_deterministic_mode_and_guards_the_other_paths():
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.engine import FineTuneTrainer, FusedTrainer, workspace_bytes
    from ecg_denoise_b200.model import ralenet_12leads as TW
    from ecg_denoise_b200.model.transformer import TransformerBlock
    x, t = _inputs(64, 256, seed=13)
    m = _model("rw", 1)
    a = _dropin_backward(m, x, t)
    assert m._plan.last_ws_bytes == workspace_bytes(64, 256, True, _lib.RL_NET_DETERMINISTIC)
    _equal(a, _dropin_backward(m, x, t), "two backward passes of one model")
    with torch_deterministic():
        assert FusedTrainer(_model("rw", 1)).deterministic
    assert not FusedTrainer(_model("rw", 1)).deterministic

    blk = TransformerBlock(16, 4, local_enhence=True).cuda()
    xb = torch.randn(4, 128, 16, device="cuda", requires_grad=True)
    with torch_deterministic():
        y = blk(xb)
        with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
            y.backward(torch.ones_like(y))
    with torch_deterministic(warn_only=True):
        y = blk(xb)
        with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
            y.backward(torch.ones_like(y))

    nm = TW.newrale(TW.ralenet(high_level_enhence=True))
    nm.load_state_dict(SW.make_newrale_state_dict(2023), strict=True)
    nm = nm.cuda().train()
    tr = FineTuneTrainer(nm, lr=1e-3)
    x12 = torch.randn(4, 12, 256, device="cuda")
    with torch_deterministic():
        with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
            tr.step(x12, x12)
    assert not torch.are_deterministic_algorithms_enabled()
