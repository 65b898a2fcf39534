"""CPU: the float64 block reference (tests/block_reference.py) that the GPU block-variant tests compare against.

  * at RL_F_PRENORM | RL_F_RESIDUAL it equals the oracle's hand-written forward and backward (oracle/ralenet_oracle.py),
    which tests/golden pins to the reference itself;
  * when the reference sources are present (oracle/ref_loader.py), it equals the reference's own float64 modules at
    every other flag: MSAttention, Mlp, TransformerBlock.forward_part1 / forward_part2 / forward and
    RelativePositionEmbedding.forward(R_pos).
"""
import contextlib
import io

import numpy as np
import pytest
import torch

from oracle import ralenet_oracle as O
from tests import block_reference as R

TOL = 1e-12


def _close(name, got, ref, tol=TOL):
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    err = float((got - ref).abs().max()) / (1.0 + float(ref.abs().max()))
    assert err <= tol, f"{name}: {err:.3e}"


def _rand(rs, *shape, scale=1.0):
    return torch.from_numpy(rs.standard_normal(shape) * scale)


def test_flag_values_match_the_c_abi():
    from ecg_denoise_b200 import _lib
    assert (R.PRENORM, R.RESIDUAL) == (_lib.CONSTS["RL_F_PRENORM"], _lib.CONSTS["RL_F_RESIDUAL"])
    assert (R.LE_NONE, R.LE_PARTIAL, R.LE_DEPTHWISE) == (
        _lib.CONSTS["RL_LE_NONE"], _lib.CONSTS["RL_LE_PARTIAL"], _lib.CONSTS["RL_LE_DEPTHWISE"])


@pytest.mark.parametrize("c0", ["centre", "zero", "end"])
@pytest.mark.parametrize("stage", [0, 1, 2, 3, 4])
def test_attn_reference_equals_oracle(stage, c0):
    rs = np.random.RandomState(10 + stage)
    C, H, L = O.CHANNELS[stage], O.HEADS[stage], O.LENGTHS[stage]
    W = O.RW_WINDOW[stage] if stage < 4 else 0
    if W == 0 and c0 != "centre":
        pytest.skip("no R-wave table at stage 4")
    off = {"centre": None, "zero": 0, "end": L - W}[c0]
    p = {k: v for k, v in R.block_params(rs, C, 0).items() if k in R.ATTN_KEYS}
    table = 0.5 * _rand(rs, 2 * W - 1, H) if W else None
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    y, dx, gr = R.attn_fwd_bwd(x, p, H, R.PRENORM | R.RESIDUAL, g, table, W, off)
    y_o, saved = O.attn_block_fwd(x, p, H, table, W, off)
    dx_o, gr_o = O.attn_block_bwd(g, saved, p, H, table, W, off)
    _close("y", y, y_o)
    _close("dx", dx, dx_o)
    for k in p:
        _close(k, gr[k], gr_o[k])
    if W:
        _close("table", gr["table"], gr_o["table"])


@pytest.mark.parametrize("le", [0, 1, 2])
@pytest.mark.parametrize("stage", [0, 2, 4])
def test_ffn_reference_equals_oracle(stage, le):
    rs = np.random.RandomState(20 + 3 * stage + le)
    C, L = O.CHANNELS[stage], O.LENGTHS[stage]
    p = {k: v for k, v in R.block_params(rs, C, le).items() if k not in R.ATTN_KEYS}
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    y, dx, gr = R.ffn_fwd_bwd(x, p, le, R.PRENORM | R.RESIDUAL, g)
    y_o, saved = O.ffn_block_fwd(x, p)
    dx_o, gr_o = O.ffn_block_bwd(g, saved, p)
    _close("y", y, y_o)
    _close("dx", dx, dx_o)
    for k in p:
        _close(k, gr[k], gr_o[k].reshape(p[k].shape))


@pytest.mark.parametrize("K", [1, 3, 15])
@pytest.mark.parametrize("with_res", [False, True])
def test_eca_reference_equals_oracle(K, with_res):
    rs = np.random.RandomState(30 + K)
    x, w, g = _rand(rs, 3, 16, 8), _rand(rs, 1, 1, K, scale=0.7), _rand(rs, 3, 16, 8)
    res = _rand(rs, 3, 16, 8) if with_res else None
    y, gr = R.with_grads(lambda x, w, res: R.ref_eca(x, w, res), g, x=x, w=w, res=res)
    y_o, saved = O.eca_fwd(x, w, res)
    dx_o, dw_o = O.eca_bwd(g, saved, w)
    _close("y", y, y_o)
    _close("dx", gr["x"], dx_o)
    _close("dw", gr["w"], dw_o)
    if with_res:
        _close("dres", gr["res"], g)


def test_flags_and_options_change_the_result():
    """each flag, option and offset the GPU tests vary changes the reference output: no axis is a duplicate."""
    rs = np.random.RandomState(40)
    C, H, L, W = 16, 4, 128, 16
    p = R.block_params(rs, C, 1)
    table = 0.5 * _rand(rs, 2 * W - 1, H)
    x, extra = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    attn = {(f, c0): R.ref_attn(x, p, H, f, table, W, c0) for f in range(4) for c0 in (0, 56, L - W)}
    ffn = {(f, le, e): R.ref_ffn(x, p if le != 2 else R.block_params(rs, C, 2), le, f, extra if e else None)
           for f in range(4) for le in range(3) for e in (0, 1)}
    nobias = {k: v for k, v in p.items() if not k.startswith("attn.qkv_proj.") or k.endswith("weight")}
    attn["nobias"] = R.ref_attn(x, nobias, H, 0, table, W, 0)
    for outs in (attn, ffn):
        vals = list(outs.values())
        for i in range(len(vals)):
            for j in range(i):
                assert float((vals[i] - vals[j]).abs().max()) > 1e-3


# ------------------------------------------------------------------------------------------------------------------
# the reference's own modules (skipped when its sources are absent)

@pytest.fixture(scope="module")
def ref():
    from oracle.ref_loader import load_reference
    r = load_reference()
    if r is None:
        pytest.skip("reference sources not found (oracle/ref_loader.find_reference)")
    return r


def _load(mod, p):
    sd = mod.state_dict()
    for k in sd:
        if k in p:
            sd[k] = p[k].reshape(sd[k].shape)
    mod.load_state_dict(sd, strict=True)
    return mod


def _module_grads(mod, fn, x, g):
    x = x.clone().requires_grad_(True)
    y = fn(x)
    y.backward(g)
    grads = {k: q.grad for k, q in mod.named_parameters() if q.grad is not None}
    return y.detach(), x.grad, grads


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):      # the reference's Mlp.__init__ prints a flag
        return fn(*a, **k)


@pytest.mark.parametrize("mask", [None, "centre", "zero", "end"])
@pytest.mark.parametrize("qkv_bias", [True, False])
@pytest.mark.parametrize("stage", [0, 1, 2, 3, 4])
def test_msattention_reference_module(ref, stage, qkv_bias, mask):
    rs = np.random.RandomState(50 + stage)
    C, H, L = O.CHANNELS[stage], O.HEADS[stage], O.LENGTHS[stage]
    W = O.RW_WINDOW[stage] if stage < 4 else 2
    p = R.block_params(rs, C, 0)
    if not qkv_bias:
        p = {k: v for k, v in p.items() if k not in ("attn.qkv_proj.to_q.bias", "attn.qkv_proj.to_kv.bias")}
    T = ref.transformer
    m = _load(T.MSAttention(C, H, qkv_bias=qkv_bias).double(), {k[5:]: v for k, v in p.items() if k.startswith("attn.")})
    table, c0, dense = None, None, None
    if mask is not None:
        rw = T.RelativePositionEmbedding(W, L, H).double()
        table = 0.5 * _rand(rs, 2 * W - 1, H)
        rw.relative_position_bias_table.data.copy_(table)
        c0 = {"centre": (L - W) // 2, "zero": 0, "end": L - W}[mask]
        dense = rw() if mask == "centre" else rw(c0 + W // 2)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    y_m, dx_m, gr_m = _module_grads(m, lambda t: m(t, mask=dense), x, g)
    y, dx, gr = R.attn_fwd_bwd(x, {k: v for k, v in p.items() if k in R.ATTN_KEYS}, H, 0, g, table,
                               W if mask else 0, c0)
    _close("y", y, y_m, 1e-10)
    _close("dx", dx, dx_m, 1e-10)
    for k, v in gr_m.items():
        _close(k, gr["attn." + k], v, 1e-10)


def _block(ref, C, H, le, use_partial, use_eca, rs):
    T = ref.transformer
    blk = _quiet(T.TransformerBlock, C, H, local_enhence=le, use_partial=use_partial, use_eca=use_eca).double()
    lemode = R.LE_NONE if not le else (R.LE_PARTIAL if use_partial else R.LE_DEPTHWISE)
    p = R.block_params(rs, C, lemode)
    if use_eca:
        p["mlp.eca.conv.weight"] = _rand(rs, 1, 1, 3, scale=0.7)
    return _load(blk, p), p, lemode


@pytest.mark.parametrize("use_eca", [False, True])
@pytest.mark.parametrize("le,use_partial", [(False, True), (True, True), (True, False)])
@pytest.mark.parametrize("stage", [0, 2, 4])
def test_mlp_reference_module(ref, stage, le, use_partial, use_eca):
    rs = np.random.RandomState(60 + stage)
    C, H, L = O.CHANNELS[stage], O.HEADS[stage], O.LENGTHS[stage]
    blk, p, lemode = _block(ref, C, H, le, use_partial, use_eca, rs)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    y_m, dx_m, gr_m = _module_grads(blk, blk.mlp, x, g)

    def fn(x, **q):
        y = R.ref_ffn(x, q, lemode, 0)
        return R.ref_eca(y, q["mlp.eca.conv.weight"]) if use_eca else y
    y, gr = R.with_grads(fn, g, x=x, **{k: v for k, v in p.items() if k.startswith("mlp.")})
    _close("y", y, y_m, 1e-10)
    _close("dx", gr["x"], dx_m, 1e-10)
    for k, v in gr_m.items():
        _close(k, gr[k], v, 1e-10)


@pytest.mark.parametrize("part", ["part1", "part2", "forward"])
@pytest.mark.parametrize("use_eca", [False, True])
@pytest.mark.parametrize("stage", [1, 3])
def test_transformer_block_reference_module(ref, stage, use_eca, part):
    rs = np.random.RandomState(70 + stage)
    C, H, L, W = O.CHANNELS[stage], O.HEADS[stage], O.LENGTHS[stage], O.RW_WINDOW[stage]
    blk, p, lemode = _block(ref, C, H, True, True, use_eca, rs)
    rw = ref.transformer.RelativePositionEmbedding(W, L, H).double()
    table = 0.5 * _rand(rs, 2 * W - 1, H)
    rw.relative_position_bias_table.data.copy_(table)
    c0 = 3
    mask = rw(c0 + W // 2)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    call = {"part1": lambda t: blk.forward_part1(t, mask), "part2": blk.forward_part2,
            "forward": lambda t: blk(t, mask)}[part]
    y_m, dx_m, gr_m = _module_grads(blk, call, x, g)

    def ffn(t, q, flags):
        if use_eca:
            return R.ref_eca(R.ref_ffn(t, q, lemode, R.PRENORM), q["mlp.eca.conv.weight"],
                             t if flags & R.RESIDUAL else None)
        return R.ref_ffn(t, q, lemode, flags)

    def fn(x, table, **q):
        if part == "part1":
            return R.ref_attn(x, q, H, R.PRENORM, table, W, c0)
        if part == "part2":
            return ffn(x, q, R.PRENORM)
        return ffn(R.ref_attn(x, q, H, R.PRENORM | R.RESIDUAL, table, W, c0), q, R.PRENORM | R.RESIDUAL)
    y, gr = R.with_grads(fn, g, x=x, table=table, **p)
    _close("y", y, y_m, 1e-10)
    _close("dx", gr["x"], dx_m, 1e-10)
    for k, v in gr_m.items():
        _close(k, gr[k], v, 1e-10)
