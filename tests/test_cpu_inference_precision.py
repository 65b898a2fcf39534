"""TF32 inference precision without a GPU: the C ABI constants, the workspace size and the module attribute."""
import copy
import pickle

import pytest

from ecg_denoise_b200 import _lib

SHAPES = [(1, 256), (515, 256), (4096, 256), (64, 512)]


def test_header_constants():
    assert _lib.RL_NET_TF32 == 2
    assert _lib.RL_F_TF32 == 4
    assert _lib.RL_NET_DETERMINISTIC == 1 and _lib.RL_F_PRENORM == 1 and _lib.RL_F_RESIDUAL == 2
    assert _lib.RL_ABI_VERSION == 4


@pytest.mark.parametrize("B,L0", SHAPES)
def test_workspace_does_not_depend_on_the_flag(B, L0):
    lib = _lib.load()
    for save in (0, 1):
        base = int(lib.ralenet_net_workspace_bytes_ex(B, L0, save, 0))
        assert int(lib.ralenet_net_workspace_bytes_ex(B, L0, save, _lib.RL_NET_TF32)) == base
        det = int(lib.ralenet_net_workspace_bytes_ex(B, L0, save, _lib.RL_NET_DETERMINISTIC))
        both = _lib.RL_NET_DETERMINISTIC | _lib.RL_NET_TF32
        assert int(lib.ralenet_net_workspace_bytes_ex(B, L0, save, both)) == det


def _models():
    from ecg_denoise_b200.model import ralenet_12leads, raletransformer, transformer
    return [transformer.ralenet(high_level_enhence=True), raletransformer.ralenet(), ralenet_12leads.ralenet()]


def test_default_is_fp32():
    for m in _models():
        assert m.inference_precision == "fp32"


@pytest.mark.parametrize("bad", ["bf16", "TF32", "", None, 32, "fp16"])
def test_bad_precision_raises(bad):
    from ecg_denoise_b200 import inference
    from ecg_denoise_b200.model import transformer
    m = transformer.ralenet()
    with pytest.raises(ValueError):
        m.inference_precision = bad
    assert m.inference_precision == "fp32"
    if bad is not None:                       # None means "keep each module's setting" in denoise_records
        with pytest.raises(ValueError):
            inference.denoise_records(m, None, precision=bad)


def test_attribute_survives_copies_and_is_not_state():
    from ecg_denoise_b200.model import transformer
    m = transformer.ralenet(high_level_enhence=True)
    keys = list(m.state_dict().keys())
    m.inference_precision = "tf32"
    assert list(m.state_dict().keys()) == keys
    assert copy.deepcopy(m).inference_precision == "tf32"
    assert pickle.loads(pickle.dumps(m)).inference_precision == "tf32"
    m.inference_precision = "fp32"
    assert copy.deepcopy(m).inference_precision == "fp32"
