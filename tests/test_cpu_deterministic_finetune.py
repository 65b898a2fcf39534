"""Deterministic 12-lead fine-tuning without a GPU: the convolution slab ABI, its argument checks and the torch-flag
resolution of FineTuneTrainer."""
import ctypes

import pytest
import torch

from ecg_denoise_b200 import _lib

# newrale's lead-mixing convolutions (Cin, Cout, K): 12 -> 6 -> 2 in front of the core, 2 -> 6 -> 12 behind it
LAYERS = [(12, 6, 13), (6, 2, 13), (2, 6, 13), (6, 12, 13)]


def _slab_bytes(B, Ci, Co, K):
    return int(_lib.load().ralenet_conv1d_slab_bytes(B, Ci, Co, K))


def test_new_symbols_are_declared_and_exported():
    lib = _lib.load()
    for name in ("ralenet_conv1d_slab_bytes", "ralenet_conv1d_bwd_det"):
        assert name in _lib.FUNCTIONS
        assert getattr(lib, name) is not None
    assert _lib.RL_ABI_VERSION == 4 and lib.ralenet_abi_version() == 4


@pytest.mark.parametrize("B", [1, 2, 37, 256, 1280, 4096])
@pytest.mark.parametrize("Ci,Co,K", LAYERS)
def test_slab_bytes_formula(B, Ci, Co, K):
    r16 = lambda n: (n + 3) // 4 * 4
    assert _slab_bytes(B, Ci, Co, K) == 4 * (r16(B * Co * Ci * K) + r16(B * Co))
    # for these shapes Co*Ci*K is a multiple of 4, so the two regions pack to one 16-byte-rounded block
    assert _slab_bytes(B, Ci, Co, K) == 4 * r16(B * (Co * Ci * K + Co))


def test_slab_bytes_of_the_whole_finetune():
    # 2,210 floats per window: the four layers' weights and biases
    assert sum(_slab_bytes(1280, *s) for s in LAYERS) == 1280 * 2210 * 4
    assert _slab_bytes(0, 12, 6, 13) == 0 and _slab_bytes(4, 12, -1, 13) == 0


def test_det_entry_point_rejects_a_null_or_short_slab_before_any_launch():
    lib = _lib.load()
    a = _lib.STRUCTS["rl_conv_bwd_args"]()
    a.B, a.L, a.Cin, a.Cout, a.K, a.act, a.slope = 37, 256, 12, 6, 13, 1, 0.01
    a.dy = a.x = a.w = a.b = a.d_w = a.d_b = 256          # never dereferenced: the checks come first
    need = _slab_bytes(37, 12, 6, 13)
    assert lib.ralenet_conv1d_bwd_det(ctypes.byref(a), None, need, None) == _lib.RL_ERR_NULL
    assert b"slab" in lib.ralenet_last_error()
    assert lib.ralenet_conv1d_bwd_det(ctypes.byref(a), 256, need - 4, None) == _lib.RL_ERR_SHAPE
    assert lib.ralenet_conv1d_bwd_det(None, 256, need, None) == _lib.RL_ERR_NULL
    a.K = 15
    assert lib.ralenet_conv1d_bwd_det(ctypes.byref(a), 256, need, None) == _lib.RL_ERR_SHAPE


def _restore(state):
    torch.use_deterministic_algorithms(state[0], warn_only=state[1])


def test_finetune_trainer_resolves_deterministic_from_the_torch_flag():
    from ecg_denoise_b200.engine import FineTuneTrainer
    from ecg_denoise_b200.model import ralenet_12leads as TW
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    state = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    try:
        torch.use_deterministic_algorithms(False)
        assert not FineTuneTrainer(m).deterministic
        assert FineTuneTrainer(m, deterministic=True).net_flags == _lib.RL_NET_DETERMINISTIC
        torch.use_deterministic_algorithms(True)
        tr = FineTuneTrainer(m)
        assert tr.deterministic and tr.net_flags == _lib.RL_NET_DETERMINISTIC
        assert not FineTuneTrainer(m, deterministic=False).deterministic
    finally:
        _restore(state)
