"""Deterministic mode without a GPU: workspace sizes of the C ABI and the torch-flag helper."""
import warnings

import pytest
import torch

from ecg_denoise_b200 import _lib

SHAPES = [(1, 256), (7, 256), (256, 256), (515, 256), (4096, 256), (64, 512), (256, 512)]


def _ws(B, L0, save, flags=None):
    lib = _lib.load()
    if flags is None:
        return int(lib.ralenet_net_workspace_bytes(B, L0, save))
    return int(lib.ralenet_net_workspace_bytes_ex(B, L0, save, flags))


@pytest.mark.parametrize("B,L0", SHAPES)
def test_workspace_ex_without_flags_equals_default(B, L0):
    for save in (0, 1):
        assert _ws(B, L0, save, 0) == _ws(B, L0, save)


@pytest.mark.parametrize("B,L0", SHAPES)
def test_deterministic_workspace_is_larger_and_a_function_of_shape(B, L0):
    det = _ws(B, L0, 1, _lib.RL_NET_DETERMINISTIC)
    assert det > _ws(B, L0, 1, 0)
    assert det % 256 == 0
    # inference (save = 0) has no backward and no partial slabs
    assert _ws(B, L0, 0, _lib.RL_NET_DETERMINISTIC) == _ws(B, L0, 0, 0)
    # the kernel-selection switches do not change the size
    lib = _lib.load()
    prev = lib.ralenet_set_wgrad_reg(2)
    try:
        assert _ws(B, L0, 1, _lib.RL_NET_DETERMINISTIC) == det
        lib.ralenet_set_wgrad_reg(0)
        prev_u = lib.ralenet_set_wgrad_umma(0)
        assert _ws(B, L0, 1, _lib.RL_NET_DETERMINISTIC) == det
        lib.ralenet_set_wgrad_umma(prev_u)
    finally:
        lib.ralenet_set_wgrad_reg(prev)


def test_deterministic_workspace_grows_with_the_batch():
    sizes = [_ws(B, 256, 1, _lib.RL_NET_DETERMINISTIC) - _ws(B, 256, 1, 0) for B in (64, 256, 1024, 4096)]
    assert sizes == sorted(sizes) and sizes[0] < sizes[-1]


def _restore(state):
    torch.use_deterministic_algorithms(state[0], warn_only=state[1])


def test_deterministic_guard_follows_the_torch_flag():
    state = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    try:
        torch.use_deterministic_algorithms(False)
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            _lib.deterministic_guard("op")                    # off: nothing happens
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
            _lib.deterministic_guard("op")
        torch.use_deterministic_algorithms(True, warn_only=True)
        with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
            _lib.deterministic_guard("op")
    finally:
        _restore(state)
    assert torch.are_deterministic_algorithms_enabled() == state[0]


def test_net_cfg_has_flags_and_mse_args_has_partials():
    cfg = _lib.STRUCTS["rl_net_cfg"]
    names = [f[0] for f in cfg._fields_]
    assert "flags" in names and "_pad" not in names
    assert names.index("flags") == names.index("save") + 1          # the old _pad slot: same layout
    assert "partials" in [f[0] for f in _lib.STRUCTS["rl_mse_args"]._fields_]
    assert _lib.RL_ABI_VERSION == 4
